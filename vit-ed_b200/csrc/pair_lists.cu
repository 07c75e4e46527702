// Index work of vited_score_pairs (engine.cu score_pairs_impl): validate a caller's pair list, find its distinct
// context and decoder items, and bucket the pairs by cell (K/V block of context slots, window of decoder slots) with a
// stable counting sort. Everything runs on the device; the caller copies the small info block back once.
//
// The counting sort works on tiles of T consecutive pairs, one warp per tile. A warp walks its tile in rounds of 32
// pairs in input order; __match_any_sync groups the lanes of a round by cell, so a group's leader can count (pass 1)
// or claim (pass 2) the group's positions in one step and every lane's rank is the number of its peers on lower
// lanes. Pass 1 writes the histogram hist[cell * tiles + tile]; its exclusive scan, cell-major, is the first output
// position of every (cell, tile); pass 2 advances those positions. Within a cell the pairs therefore keep their input
// order: the same list always gives the same chunks.
#include "kernels.h"

namespace vited {

// ------------------------------------------------------------------------------------------------------------
// mark + validate: used[a] (context) / used[N + b] (decoder) = 1; indices outside [0, N) are counted and the lowest
// offending pair is kept (info[PL_FIRST_BAD] starts at 0xffffffff).
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) pairs_mark_kernel(const int* __restrict__ pairs, int P, int N,
                                                         int* __restrict__ used, int* __restrict__ info) {
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < P; p += (int64_t)gridDim.x * blockDim.x) {
    const int a = pairs[2 * p], b = pairs[2 * p + 1];
    if (a < 0 || a >= N || b < 0 || b >= N) {
      atomicAdd(&info[PL_N_BAD], 1);
      atomicMin(reinterpret_cast<unsigned*>(&info[PL_FIRST_BAD]), (unsigned)p);
    } else {
      used[a] = 1;
      used[N + b] = 1;
    }
  }
}

int pairs_mark(const int* pairs, int P, int N, int* used, int* info, cudaStream_t stream) {
  if (P == 0) return 0;
  int blocks = (int)(((int64_t)P + 255) / 256);
  if (blocks > 148 * 16) blocks = 148 * 16;
  pairs_mark_kernel<<<blocks, 256, 0, stream>>>(pairs, P, N, used, info);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------------------
// exclusive prefix sum of n ints in one block (n is at most a few million here: N flags, or cells x tiles), in place
// allowed; *total = sum. Every thread scans 8 consecutive values per round, warps combine through shared memory.
// ------------------------------------------------------------------------------------------------------------
constexpr int SCAN_THREADS = 1024;
constexpr int SCAN_ITEMS = 8;

__global__ void __launch_bounds__(SCAN_THREADS) exclusive_scan_kernel(const int* in, int* out, int64_t n, int* total) {
  __shared__ int warp_off[SCAN_THREADS / 32];
  __shared__ int carry;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int64_t base = 0; base < n; base += (int64_t)SCAN_THREADS * SCAN_ITEMS) {
    const int64_t i0 = base + (int64_t)threadIdx.x * SCAN_ITEMS;
    int v[SCAN_ITEMS];
    int sum = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) {
      v[k] = (i0 + k < n) ? in[i0 + k] : 0;
      sum += v[k];
    }
    int incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane == 31) warp_off[warp] = incl;
    __syncthreads();
    if (warp == 0) {
      const int w = warp_off[lane];
      int wi = w;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, wi, o);
        if (lane >= o) wi += t;
      }
      warp_off[lane] = wi - w;
    }
    __syncthreads();
    int run = carry + warp_off[warp] + incl - sum;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) {
      if (i0 + k < n) out[i0 + k] = run;
      run += v[k];
    }
    __syncthreads();                                    // every thread has read carry and warp_off
    if (threadIdx.x == SCAN_THREADS - 1) carry = run;   // the last thread's running sum ends the round
    __syncthreads();
  }
  if (threadIdx.x == 0) *total = carry;
}

int exclusive_scan(const int* in, int* out, int64_t n, int* total, cudaStream_t stream) {
  exclusive_scan_kernel<<<1, SCAN_THREADS, 0, stream>>>(in, out, n, total);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------------------
// compact: items[slot[i]] = i for every used i, separately for the context half [0, N) and the decoder half [N, 2N)
// of used / slot / items (ascending item lists; slot is the exclusive scan of used within each half)
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) pairs_compact_kernel(const int* __restrict__ used, const int* __restrict__ slot,
                                                            int* __restrict__ items, int N) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < 2 * (int64_t)N; i += (int64_t)gridDim.x * blockDim.x) {
    if (!used[i]) continue;
    const int half = i >= N ? 1 : 0;
    items[(int64_t)half * N + slot[i]] = (int)(i - (int64_t)half * N);
  }
}

int pairs_compact(const int* used, const int* slot, int* items, int N, cudaStream_t stream) {
  if (N == 0) return 0;
  int blocks = (int)((2 * (int64_t)N + 255) / 256);
  if (blocks > 148 * 16) blocks = 148 * 16;
  pairs_compact_kernel<<<blocks, 256, 0, stream>>>(used, slot, items, N);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------------------
// counting sort by cell (see the top of the file). cell = (ctx slot / rb) * nw + decoder slot / cw; -1 for lanes past
// the tile and for invalid pairs (those make the call fail before any scoring, they only must not be indexed).
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int pair_cell(const int* __restrict__ pairs, int64_t p, int N, const int* __restrict__ slot,
                                         const PairCells& c, int* ctx_slot, int* x2_slot) {
  const int a = pairs[2 * p], b = pairs[2 * p + 1];
  if (a < 0 || a >= N || b < 0 || b >= N) return -1;
  *ctx_slot = slot[a];
  *x2_slot = slot[N + b];
  return (*ctx_slot / c.rb) * c.nw + *x2_slot / c.cw;
}

template <bool SCATTER>
__global__ void __launch_bounds__(256) pairs_bucket_kernel(const int* __restrict__ pairs, int P, int N,
                                                           const int* __restrict__ slot, PairCells c, int* hist,
                                                           int* __restrict__ ci, int* __restrict__ xj,
                                                           int* __restrict__ out_pos) {
  const int lane = threadIdx.x & 31;
  const int tile = (int)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (tile >= c.tiles) return;                          // warp-uniform
  const int64_t p0 = (int64_t)tile * c.T;
  const int64_t p1 = p0 + c.T < P ? p0 + c.T : P;
  for (int64_t base = p0; base < p1; base += 32) {
    const int64_t p = base + lane;
    int cs = 0, xs = 0;
    const int cell = p < p1 ? pair_cell(pairs, p, N, slot, c, &cs, &xs) : -1;
    const unsigned peers = __match_any_sync(0xffffffffu, cell);
    const int leader = __ffs(peers) - 1;
    int* counter = cell >= 0 ? hist + (size_t)cell * c.tiles + tile : nullptr;
    if (!SCATTER) {
      if (cell >= 0 && lane == leader) *counter += __popc(peers);
    } else {
      int first = 0;
      if (cell >= 0 && lane == leader) first = *counter;
      first = __shfl_sync(0xffffffffu, first, leader);
      if (cell >= 0) {
        const int pos = first + __popc(peers & ((1u << lane) - 1u));
        ci[pos] = cs % c.rb;
        xj[pos] = xs;
        out_pos[pos] = (int)p;
        if (lane == leader) *counter = first + __popc(peers);
      }
    }
    __syncwarp();                                       // the next round's leader of a cell may be another lane
  }
}

int pairs_bucket_count(const int* pairs, int P, int N, const int* slot, const PairCells& c, int* hist,
                       cudaStream_t stream) {
  const int blocks = (c.tiles + 7) / 8;
  pairs_bucket_kernel<false><<<blocks, 256, 0, stream>>>(pairs, P, N, slot, c, hist, nullptr, nullptr, nullptr);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}

int pairs_bucket_scatter(const int* pairs, int P, int N, const int* slot, const PairCells& c, int* hist, int* ci,
                         int* xj, int* out_pos, cudaStream_t stream) {
  const int blocks = (c.tiles + 7) / 8;
  pairs_bucket_kernel<true><<<blocks, 256, 0, stream>>>(pairs, P, N, slot, c, hist, ci, xj, out_pos);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}

// info[PL_CELLS + k] = first sorted position of cell k (hist scanned, before the scatter advances it); the offending
// pair's two indices when there is one
__global__ void pairs_cell_starts_kernel(const int* __restrict__ pairs, const int* __restrict__ hist, int tiles,
                                         int cells, int* __restrict__ info) {
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < cells; k += gridDim.x * blockDim.x)
    info[PL_CELLS + k] = hist[(size_t)k * tiles];
  if (blockIdx.x == 0 && threadIdx.x == 0 && info[PL_N_BAD] > 0) {
    const size_t f = (unsigned)info[PL_FIRST_BAD];
    info[PL_BAD_A] = pairs[2 * f];
    info[PL_BAD_B] = pairs[2 * f + 1];
  }
}

int pairs_cell_starts(const int* pairs, const int* hist, int tiles, int cells, int* info, cudaStream_t stream) {
  int blocks = (cells + 255) / 256;
  if (blocks > 148 * 4) blocks = 148 * 4;
  pairs_cell_starts_kernel<<<blocks, 256, 0, stream>>>(pairs, hist, tiles, cells, info);
  VITED_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // namespace vited
