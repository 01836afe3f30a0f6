// spn_track_labels / spn_track_table (include/spn_tracks.h): connected components of the match graph by union-find
// after ECL-CC (Jaiganesh & Burtscher 2018), and the track table from the component labels.
//
// Labels.  label[] is the union-find forest itself: every row points at a row of its component that is no larger, a
// root points at itself.  A hook only ever writes a root, with atomicCAS, and only under a smaller root; finds halve
// their path with plain stores, which only ever replace a pointer by one of its ancestors.  So a component's root is
// its minimum row, whatever order the hooks land in.  After the hooks, rounds of pointer jumping make every row point
// at its root: a round halves every path, so bits(K) rounds suffice for any depth (a chain fed in descending order is
// the deepest case), and a round that changes nothing makes the later rounds return at once.
//
// Table.  Component sizes by integer atomics; one exclusive scan over the roots of (is track << 32 | size) gives every
// track its index (high word) and its first observation (low word, O <= K < 2^31); a stable radix sort of the rows by
// track index puts each track's rows in ascending order, so no atomic decides the observation order.
#include <algorithm>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "spn_common.cuh"
#include "../../include/spn_tracks.h"

namespace {

constexpr int kThreads = 256;
constexpr int kMaxRounds = 32;  // bits(K) <= 31 pointer-jumping rounds, plus room

__device__ __forceinline__ int find_halving(volatile int* lab, int x) {
  int cur = lab[x];
  if (cur != x) {
    int prev = x, next;
    while (cur > (next = lab[cur])) {
      lab[prev] = next;
      prev = cur;
      cur = next;
    }
  }
  return cur;
}

__global__ void __launch_bounds__(kThreads) labels_init_kernel(int* __restrict__ lab, int K, int resume,
                                                               unsigned long long* __restrict__ bad) {
  for (long long rr = blockIdx.x * (long long)blockDim.x + threadIdx.x; rr < K; rr += (long long)gridDim.x * blockDim.x) {
    const int r = (int)rr;
    if (!resume) {
      lab[r] = r;
    } else {
      const int l = lab[r];
      if (l < 0 || l > r) {
        lab[r] = r;
        atomicAdd(bad, 1ull);
      }
    }
  }
}

__global__ void __launch_bounds__(kThreads) labels_hook_kernel(const int* __restrict__ edges, long long E, int* lab, int K,
                                                               unsigned long long* __restrict__ bad) {
  volatile int* vl = lab;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < E; e += (long long)gridDim.x * blockDim.x) {
    const int u = __ldg(edges + 2 * e), v = __ldg(edges + 2 * e + 1);
    if (u < 0 || u >= K || v < 0 || v >= K) {
      atomicAdd(bad, 1ull);
      continue;
    }
    int ru = find_halving(vl, u), rv = find_halving(vl, v);
    while (ru != rv) {  // hook the larger root under the smaller; a failed CAS returns the larger one's new parent
      if (ru < rv) {
        const int old = atomicCAS(lab + rv, rv, ru);
        if (old == rv) break;
        rv = find_halving(vl, old);
      } else {
        const int old = atomicCAS(lab + ru, ru, rv);
        if (old == ru) break;
        ru = find_halving(vl, old);
      }
    }
  }
}

// One round of pointer jumping; returns at once when the previous round changed nothing (round 0 always runs).
__global__ void __launch_bounds__(kThreads) labels_jump_kernel(int* lab, int K, int* __restrict__ changed, int round) {
  if (round > 0 && *(volatile int*)(changed + round - 1) == 0) return;
  volatile int* vl = lab;
  bool any = false;
  for (long long rr = blockIdx.x * (long long)blockDim.x + threadIdx.x; rr < K; rr += (long long)gridDim.x * blockDim.x) {
    const int r = (int)rr;
    const int l = vl[r], ll = vl[l];
    if (ll != l) {
      vl[r] = ll;
      any = true;
    }
  }
  if (__syncthreads_or(any) && threadIdx.x == 0) changed[round] = 1;
}

struct TableParams {
  const int* label;
  const long long* img_off;
  int K, N, min_length, sentinel;
  int* size_keys;              // [K] component sizes, then the sort keys (track index, or sentinel)
  unsigned long long* scan_in; // [K] (is track << 32 | size) at the roots; later the sorted keys / rows
  unsigned long long* scan_out;
  int* rows;                   // [K] 0 .. K-1, the sort's values
  long long* track_off;
  int* obs;
  unsigned char* consistent;
  int* track_of;
  long long* totals;
  unsigned long long* bad;
};

// A label of spn_track_labels: in [0, r] and pointing at a root.
__device__ __forceinline__ bool valid_label(const int* lab, int r, int l) { return l >= 0 && l <= r && lab[l] == l; }

__global__ void __launch_bounds__(kThreads) table_count_kernel(TableParams p) {
  const int n_items = max(p.K, p.N);
  for (long long rr = blockIdx.x * (long long)blockDim.x + threadIdx.x; rr < n_items; rr += (long long)gridDim.x * blockDim.x) {
    const int r = (int)rr;
    if (r < p.K) {
      const int l = p.label[r];
      if (valid_label(p.label, r, l)) atomicAdd(p.size_keys + l, 1);
      else atomicAdd(p.bad, 1ull);
    }
    if (r < p.N) {
      bool ok = p.img_off[r] <= p.img_off[r + 1];
      if (r == 0) ok = ok && p.img_off[0] == 0 && p.img_off[p.N] == p.K;
      if (!ok) atomicAdd(p.bad, 1ull);
    }
  }
}

__global__ void __launch_bounds__(kThreads) table_flag_kernel(TableParams p) {
  for (long long rr = blockIdx.x * (long long)blockDim.x + threadIdx.x; rr < p.K; rr += (long long)gridDim.x * blockDim.x) {
    const int r = (int)rr;
    const int sz = p.size_keys[r];
    p.scan_in[r] = (p.label[r] == r && sz >= p.min_length) ? (1ull << 32) | (unsigned)sz : 0ull;
  }
}

__global__ void __launch_bounds__(kThreads) table_assign_kernel(TableParams p) {
  for (long long rr = blockIdx.x * (long long)blockDim.x + threadIdx.x; rr < p.K; rr += (long long)gridDim.x * blockDim.x) {
    const int r = (int)rr;
    const int l = p.label[r];
    int t = -1;
    if (valid_label(p.label, r, l) && p.scan_in[l] != 0ull) t = (int)(p.scan_out[l] >> 32);
    p.track_of[r] = t;
    p.size_keys[r] = t >= 0 ? t : p.sentinel;
    p.rows[r] = r;
    if (t >= 0 && l == r) {
      p.track_off[t] = (long long)(p.scan_out[r] & 0xffffffffull);
      p.consistent[t] = 1;
    }
    if (r == p.K - 1) {
      const unsigned long long end = p.scan_out[r] + p.scan_in[r];
      const long long T = (long long)(end >> 32), O = (long long)(end & 0xffffffffull);
      p.totals[0] = T;
      p.totals[1] = O;
      p.track_off[T] = O;
    }
  }
}

// The image of row r: the largest n with img_off[n] <= r (skips images without keypoints).
__device__ __forceinline__ int image_of(const long long* off, int N, int r) {
  int lo = 0, hi = N - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (off[mid] <= r) lo = mid;
    else hi = mid - 1;
  }
  return lo;
}

__global__ void __launch_bounds__(kThreads) table_obs_kernel(TableParams p, const int* __restrict__ keys,
                                                             const int* __restrict__ rows) {
  const long long O = p.totals[1];
  for (long long ii = blockIdx.x * (long long)blockDim.x + threadIdx.x; ii < O; ii += (long long)gridDim.x * blockDim.x) {
    const int i = (int)ii;
    const int r = rows[i], n = image_of(p.img_off, p.N, r);
    p.obs[2 * ii] = n;
    p.obs[2 * ii + 1] = (int)(r - p.img_off[n]);
    if (i > 0 && keys[i - 1] == keys[i] && image_of(p.img_off, p.N, rows[i - 1]) == n) p.consistent[keys[i]] = 0;
  }
}

inline int grid_for(long long n, int sm_count) {
  const long long blocks = (n + kThreads - 1) / kThreads;
  return (int)std::max(1ll, std::min(blocks, (long long)sm_count * 8));
}

inline size_t align256(size_t x) { return (x + 255) & ~size_t(255); }

}  // namespace

extern "C" int spn_track_labels(spn_ctx* ctx, const int32_t* d_edges, int64_t E, int32_t K, int resume, int32_t* d_label,
                                int64_t* d_bad, spn_stream stream) {
  SPN_REQUIRE(ctx, "spn_track_labels: null pointer (ctx)");
  SPN_REQUIRE(K > 0, "spn_track_labels: K = %d rows must be in [1, 2^31 - 1]", K);
  SPN_REQUIRE(E >= 0, "spn_track_labels: E = %lld edges must be >= 0", (long long)E);
  SPN_REQUIRE(resume == 0 || resume == 1, "spn_track_labels: resume = %d must be 0 or 1", resume);
  SPN_REQUIRE(E == 0 || d_edges, "spn_track_labels: null pointer (edges with E = %lld)", (long long)E);
  SPN_REQUIRE(d_label && d_bad, "spn_track_labels: null pointer (label / bad)");
  SpnDeviceGuard guard(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;
  int rc = spn_ensure_aux(ctx, kMaxRounds * sizeof(int), s);
  if (rc) return rc;
  int* changed = (int*)ctx->aux;
  SPN_CUDA(cudaMemsetAsync(changed, 0, kMaxRounds * sizeof(int), s));
  SPN_CUDA(cudaMemsetAsync(d_bad, 0, sizeof(int64_t), s));
  unsigned long long* bad = (unsigned long long*)d_bad;
  const int gk = grid_for(K, ctx->sm_count);
  labels_init_kernel<<<gk, kThreads, 0, s>>>(d_label, K, resume, bad);
  SPN_CHECK_LAUNCH(ctx);
  if (E > 0) {
    labels_hook_kernel<<<grid_for(E, ctx->sm_count), kThreads, 0, s>>>(d_edges, E, d_label, K, bad);
    SPN_CHECK_LAUNCH(ctx);
  }
  const int rounds = 32 - __builtin_clz((unsigned)K);  // bits(K): halving a path of at most K - 1 steps
  for (int i = 0; i < rounds; ++i) {
    labels_jump_kernel<<<gk, kThreads, 0, s>>>(d_label, K, changed, i);
    SPN_CHECK_LAUNCH(ctx);
  }
  return SPN_OK;
}

extern "C" int spn_track_table(spn_ctx* ctx, const int32_t* d_label, int32_t K, const int64_t* d_img_offsets, int32_t N,
                               int32_t min_length, int64_t* d_track_offsets, int32_t* d_obs, uint8_t* d_consistent,
                               int32_t* d_track_of, int64_t* d_totals, int64_t* d_bad, spn_stream stream) {
  SPN_REQUIRE(ctx, "spn_track_table: null pointer (ctx)");
  SPN_REQUIRE(K > 0, "spn_track_table: K = %d rows must be in [1, 2^31 - 1]", K);
  SPN_REQUIRE(N > 0 && N < 0x7fffffff, "spn_track_table: N = %d images must be in [1, 2^31 - 2]", N);
  SPN_REQUIRE(min_length >= 2, "spn_track_table: min_length = %d must be >= 2", min_length);
  SPN_REQUIRE(d_label && d_img_offsets && d_track_offsets && d_obs && d_track_of && d_totals && d_bad,
              "spn_track_table: null pointer (label / img_offsets / track_offsets / obs / track_of / totals / bad)");
  SPN_REQUIRE(K < 2 || d_consistent, "spn_track_table: null pointer (consistent with K = %d)", K);
  SpnDeviceGuard guard(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;
  const int sentinel = K / 2;  // > every track index, since T <= K / 2
  const int end_bit = std::max(1, 32 - __builtin_clz((unsigned)std::max(sentinel, 1)));
  size_t scan_tmp = 0, sort_tmp = 0;
  SPN_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, scan_tmp, (unsigned long long*)nullptr, (unsigned long long*)nullptr, K, s));
  SPN_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, sort_tmp, (const int*)nullptr, (int*)nullptr, (const int*)nullptr,
                                           (int*)nullptr, K, 0, end_bit, s));
  const size_t b4 = align256((size_t)K * 4), b8 = align256((size_t)K * 8);
  const size_t tmp = align256(std::max(scan_tmp, sort_tmp));
  int rc = spn_ensure_aux(ctx, b4 + 2 * b8 + b4 + tmp, s);
  if (rc) return rc;
  char* base = ctx->aux;
  TableParams p;
  p.label = d_label; p.img_off = (const long long*)d_img_offsets; p.K = K; p.N = N; p.min_length = min_length;
  p.sentinel = sentinel;
  p.size_keys = (int*)base;
  p.scan_in = (unsigned long long*)(base + b4);
  p.scan_out = (unsigned long long*)(base + b4 + b8);
  p.rows = (int*)(base + b4 + 2 * b8);
  void* temp = base + 2 * b4 + 2 * b8;
  p.track_off = (long long*)d_track_offsets; p.obs = d_obs; p.consistent = d_consistent; p.track_of = d_track_of;
  p.totals = (long long*)d_totals; p.bad = (unsigned long long*)d_bad;
  // after the scan, scan_in's storage holds the sorted keys and rows (K int32 each)
  int* keys_out = (int*)p.scan_in;
  int* rows_out = keys_out + K;
  SPN_CUDA(cudaMemsetAsync(p.size_keys, 0, (size_t)K * 4, s));
  SPN_CUDA(cudaMemsetAsync(d_bad, 0, sizeof(int64_t), s));
  const int g = grid_for(std::max(K, N), ctx->sm_count);
  table_count_kernel<<<g, kThreads, 0, s>>>(p);
  SPN_CHECK_LAUNCH(ctx);
  table_flag_kernel<<<g, kThreads, 0, s>>>(p);
  SPN_CHECK_LAUNCH(ctx);
  SPN_CUDA(cub::DeviceScan::ExclusiveSum(temp, scan_tmp, p.scan_in, p.scan_out, K, s));
  table_assign_kernel<<<g, kThreads, 0, s>>>(p);
  SPN_CHECK_LAUNCH(ctx);
  SPN_CUDA(cub::DeviceRadixSort::SortPairs(temp, sort_tmp, (const int*)p.size_keys, keys_out, (const int*)p.rows, rows_out, K, 0,
                                           end_bit, s));
  table_obs_kernel<<<g, kThreads, 0, s>>>(p, keys_out, rows_out);
  SPN_CHECK_LAUNCH(ctx);
  return SPN_OK;
}
