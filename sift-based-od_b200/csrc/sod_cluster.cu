// Pose clustering after the affine stage (SURVEY.md §8f N1): the O(V^2) neighbour tests of
// group_position (PostProcessing.py:14-37) and group_orientation (PostProcessing.py:39-63) as bit
// matrices, plus the connected components of each graph by a lock-free union-find.  The depth-first
// visiting order that fixes the reference's float summation order is recovered on the host from the
// bit rows (sod_b200/postprocess.py); the pair tests themselves use the reference's fp64 expressions.
//
// sod_final_poses runs all four steps of Main.post_process (group_position -> group_orientation ->
// find_max_orientation -> get_final_pose) on the device, with no host step between the bins and the poses:
// bins sorted by segment (stable), the position bit rows of every segment, one warp per segment walking the
// depth-first pre-order, the orientation bit rows of every cluster, one warp per cluster walking its
// sub-clusters and summing in visiting order, and one CTA numbering the clusters by their lowest bin.
#include <cub/block/block_scan.cuh>

#include "sod_common.cuh"

namespace sod {
namespace {

constexpr int kThreads = 256;

// The pair tests of the two neighbour graphs, shared by adjacency_kernel and the final-pose kernels below.
// group_position (PostProcessing.py:17-30): abs(xa - xb) <= w_a*s_a/4 and abs(ya - yb) <= h_a*s_a/4 and the same
// against bin b (reach = img_size * scale / 4, pose_reach).
__device__ __forceinline__ bool position_edge(double xa, double ya, double rxa, double rya, double xb, double yb,
                                              double rxb, double ryb) {
  const double dx = fabs(__dsub_rn(xb, xa)), dy = fabs(__dsub_rn(yb, ya));
  return dx <= rxb && dy <= ryb && dx <= rxa && dy <= rya;
}

// group_orientation (PostProcessing.py:43-56): abs(math.degrees(angle_a - angle_b)) <= max_degrees;
// math.degrees(x) is x * (180 / pi) in double.
__device__ __forceinline__ bool angle_edge(double a, double b, double max_degrees) {
  return fabs(__dmul_rn(__dsub_rn(b, a), 180.0 / 3.14159265358979323846)) <= max_degrees;
}

// img_size * scale / 4: the product rounded once, then a division by 4, which is exact scaling and so the same
// rounding as the multiplication by 0.25.
__device__ __forceinline__ double pose_reach(double size, double scale) {
  return __dmul_rn(__dmul_rn(size, scale), 0.25);
}

// Loads go to L2 (__ldcg): another SM's hook must not hide behind a stale L1 line.
__device__ __forceinline__ int uf_find(int* parent, int x) {
  int p = __ldcg(parent + x);
  while (p != x) {  // path halving; parents only ever decrease, so stale reads are still ancestors
    const int g = __ldcg(parent + p);
    if (g != p) parent[x] = g;
    x = p;
    p = __ldcg(parent + x);
  }
  return x;
}

// Roots are always hooked under the smaller root: the final root of a component is its lowest index.
__device__ __forceinline__ void uf_union(int* parent, int a, int b) {
  for (;;) {
    a = uf_find(parent, a);
    b = uf_find(parent, b);
    if (a == b) return;
    if (a < b) {
      const int t = a;
      a = b;
      b = t;
    }
    if (atomicCAS(parent + a, a, b) == a) return;
  }
}

__global__ void label_init_kernel(int* __restrict__ label, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) label[i] = i;
}

// Final labels.  No path compression here: a halving store that was computed from older parents could
// land after a thread has written its final label and replace it by a mere ancestor.  The walk only
// reads; the one store per thread writes a root, which is a valid parent for every concurrent reader.
__global__ void label_flatten_kernel(int* __restrict__ label, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int x = i, p = __ldcg(label + x);
  while (p != x) {
    x = p;
    p = __ldcg(label + x);
  }
  label[i] = x;
}

// One CTA per bin i; its warps sweep the other bins 32 at a time (lane <-> j), __ballot_sync builds the
// adjacency word.  kind 0: position test, kind 1: angle test.
template <int kKind>
__global__ void __launch_bounds__(kThreads)
adjacency_kernel(const double* __restrict__ a0, const double* __restrict__ a1, const double* __restrict__ a2,
                 const double* __restrict__ a3, const int32_t* __restrict__ segment, int n, double limit,
                 uint32_t* __restrict__ adj, int* __restrict__ parent) {
  const int i = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int words = (n + 31) >> 5;
  const int seg_i = segment ? segment[i] : 0;
  const double xi = a0[i];
  double yi = 0.0, wi = 0.0, hi = 0.0;
  if (kKind == 0) {
    yi = a1[i];
    wi = a2[i];
    hi = a3[i];
  }
  for (int w = warp; w < words; w += kThreads / 32) {
    const int j = w * 32 + lane;
    bool edge = false;
    if (j < n && j != i && (!segment || segment[j] == seg_i)) {
      if (kKind == 0) {
        edge = position_edge(xi, yi, wi, hi, a0[j], a1[j], a2[j], a3[j]);
      } else {
        edge = angle_edge(xi, a0[j], limit);
      }
    }
    const uint32_t word = __ballot_sync(0xffffffffu, edge);
    if (lane == 0) adj[static_cast<size_t>(i) * words + w] = word;
    if (edge && j < i) uf_union(parent, i, j);
  }
}

template <int kKind>
int run_adjacency(const double* a0, const double* a1, const double* a2, const double* a3, const int32_t* segment,
                  int64_t n, double limit, uint32_t* adj, int32_t* label, sod_stream_t stream) {
  SOD_CHECK_ARG(n >= 0 && n <= SOD_MAX_CLUSTER_BINS, "n must be in 0..%d", SOD_MAX_CLUSTER_BINS);
  if (n == 0) return SOD_OK;
  SOD_CHECK_ARG(a0 && adj && label && (kKind == 1 || (a1 && a2 && a3)), "null pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int ni = static_cast<int>(n);
  const unsigned blocks = static_cast<unsigned>((ni + kThreads - 1) / kThreads);
  label_init_kernel<<<blocks, kThreads, 0, st>>>(label, ni);
  SOD_CHECK_LAUNCH("label_init_kernel");
  adjacency_kernel<kKind><<<static_cast<unsigned>(ni), kThreads, 0, st>>>(a0, a1, a2, a3, segment, ni, limit, adj,
                                                                         label);
  SOD_CHECK_LAUNCH("adjacency_kernel");
  label_flatten_kernel<<<blocks, kThreads, 0, st>>>(label, ni);
  SOD_CHECK_LAUNCH("label_flatten_kernel");
  return SOD_OK;
}


// ------------------------------------------------------------------------------------------------ final poses

constexpr int kRankThreads = 256;
constexpr int kFinishThreads = 1024;
constexpr int kSortThreads = 1024, kSortWarps = kSortThreads / 32;
constexpr int kWalkGrid = 4096;                      // CTAs (one warp each) of the two walks, over the start lists
constexpr int kVisWords = SOD_MAX_CLUSTER_BINS / 32; // a walk's visited bits, in shared memory
constexpr uint32_t kKeyEnd = 0xffffffffu;           // sort key of the slots past the count
constexpr int kSmall = 32;                           // clusters of up to 32 bins: bit rows in registers

__device__ __forceinline__ uint32_t segment_key(int32_t seg) { return static_cast<uint32_t>(seg) ^ 0x80000000u; }

// Workspace views, by sorted position q (the bins ordered by segment, stable) or by bin index b.
struct PoseTmp {
  uint32_t *key_in, *key;       // segment keys: input order, sorted
  int32_t *bin_in, *bin;        // q -> b
  int32_t* count;               // [0] bins clustered, [1] live bins (records path), [2] segments, [3] clusters
  int32_t *seg_list, *cl_list;  // first position of every segment / cluster, in no particular order
  double* smean;                // records path: the live bins' means in (group, order key) order
  int32_t* sseg;                //   and their segment (frame)
  double *x, *y, *rx, *ry, *ang;  // by q
  int32_t *seg_lo, *seg_len;    // by q: the segment's first position and size
  int32_t *order, *cl_lo, *cl_len;  // by visiting position k: sorted position, cluster's first k and size
  double* oang;                 // by k: angle of order[k]
  int32_t *sub, *sub_first;     // by k: sorted positions in sub-cluster order, 1 where a sub-cluster starts
  int32_t *cursor, *stack;      // the walks' per-node word cursor and stack
  int32_t *root_size, *root_k, *root_dst, *root_shape;  // by bin b: 0 or the size of the cluster whose lowest bin is b
  double* root_pose;            // by b: [6]
  uint32_t* adj;                // bit rows; segment / cluster starting at q has rows at adj + q * words_cap
  int64_t words_cap;
};

struct PoseLayout {
  size_t key_in, key, bin_in, bin, count, seg_list, cl_list, smean, sseg, x, y, rx, ry, ang, seg_lo, seg_len, order, cl_lo, cl_len, oang,
      sub, sub_first, cursor, stack, root_size, root_k, root_dst, root_shape, root_pose, adj, total;
};

PoseLayout pose_layout(int64_t cap) {
  PoseLayout L{};
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t at = off;
    off += (bytes + 255) & ~size_t(255);
    return at;
  };
  const size_t n = static_cast<size_t>(cap > 0 ? cap : 1);
  const size_t i4 = n * 4, f8 = n * 8;
  L.key_in = take(i4); L.key = take(i4); L.bin_in = take(i4); L.bin = take(i4); L.count = take(16);
  L.seg_list = take(i4); L.cl_list = take(i4);
  L.smean = take(6 * f8); L.sseg = take(i4);
  L.x = take(f8); L.y = take(f8); L.rx = take(f8); L.ry = take(f8); L.ang = take(f8);
  L.seg_lo = take(i4); L.seg_len = take(i4); L.order = take(i4); L.cl_lo = take(i4); L.cl_len = take(i4);
  L.oang = take(f8); L.sub = take(i4); L.sub_first = take(i4); L.cursor = take(i4); L.stack = take(i4);
  L.root_size = take(i4); L.root_k = take(i4); L.root_dst = take(i4); L.root_shape = take(i4);
  L.root_pose = take(6 * f8);
  L.adj = take(n * ((n + 31) / 32) * 4);
  L.total = off;
  return L;
}

PoseTmp pose_tmp(void* ws, int64_t cap) {
  const PoseLayout L = pose_layout(cap);
  char* b = static_cast<char*>(ws);
  PoseTmp t;
  t.key_in = reinterpret_cast<uint32_t*>(b + L.key_in); t.key = reinterpret_cast<uint32_t*>(b + L.key);
  t.bin_in = reinterpret_cast<int32_t*>(b + L.bin_in); t.bin = reinterpret_cast<int32_t*>(b + L.bin);
  t.count = reinterpret_cast<int32_t*>(b + L.count);
  t.seg_list = reinterpret_cast<int32_t*>(b + L.seg_list); t.cl_list = reinterpret_cast<int32_t*>(b + L.cl_list);
  t.smean = reinterpret_cast<double*>(b + L.smean); t.sseg = reinterpret_cast<int32_t*>(b + L.sseg);
  t.x = reinterpret_cast<double*>(b + L.x); t.y = reinterpret_cast<double*>(b + L.y);
  t.rx = reinterpret_cast<double*>(b + L.rx); t.ry = reinterpret_cast<double*>(b + L.ry);
  t.ang = reinterpret_cast<double*>(b + L.ang);
  t.seg_lo = reinterpret_cast<int32_t*>(b + L.seg_lo); t.seg_len = reinterpret_cast<int32_t*>(b + L.seg_len);
  t.order = reinterpret_cast<int32_t*>(b + L.order); t.cl_lo = reinterpret_cast<int32_t*>(b + L.cl_lo);
  t.cl_len = reinterpret_cast<int32_t*>(b + L.cl_len); t.oang = reinterpret_cast<double*>(b + L.oang);
  t.sub = reinterpret_cast<int32_t*>(b + L.sub); t.sub_first = reinterpret_cast<int32_t*>(b + L.sub_first);
  t.cursor = reinterpret_cast<int32_t*>(b + L.cursor); t.stack = reinterpret_cast<int32_t*>(b + L.stack);
  t.root_size = reinterpret_cast<int32_t*>(b + L.root_size); t.root_k = reinterpret_cast<int32_t*>(b + L.root_k);
  t.root_dst = reinterpret_cast<int32_t*>(b + L.root_dst);
  t.root_shape = reinterpret_cast<int32_t*>(b + L.root_shape);
  t.root_pose = reinterpret_cast<double*>(b + L.root_pose);
  t.adj = reinterpret_cast<uint32_t*>(b + L.adj);
  t.words_cap = (cap + 31) / 32;
  return t;
}

// Optional pre-pass of the live path: the affine stage's records (status bit 0 = live) -> the live bins in
// (group, order key) order, i.e. final_poses' host lexsort by (frame, group, order key) with frame = group /
// groups_per_frame.  A bin's rank is the number of live bins with a smaller key (ties, which the Hough
// insertion keys never have, by record index).
__global__ void __launch_bounds__(kRankThreads)
live_rank_kernel(const int32_t* __restrict__ status, const int32_t* __restrict__ group,
                 const int64_t* __restrict__ order_key, const double* __restrict__ mean,
                 const int32_t* __restrict__ n_dev, int cap, int groups_per_frame, PoseTmp t) {
  __shared__ int32_t s_group[kRankThreads];
  __shared__ int64_t s_key[kRankThreads];
  __shared__ int32_t s_live[kRankThreads];
  const int count = min(max(*n_dev, 0), cap);
  const int i = blockIdx.x * kRankThreads + threadIdx.x;
  const bool live = i < count && (status[i] & 1);
  const int32_t gi = live ? group[i] : 0;
  const int64_t oi = live ? order_key[i] : 0;
  int rank = 0, total = 0;
  for (int j0 = 0; j0 < count; j0 += kRankThreads) {
    const int j = j0 + threadIdx.x;
    s_live[threadIdx.x] = j < count && (status[j] & 1);
    s_group[threadIdx.x] = j < count ? group[j] : 0;
    s_key[threadIdx.x] = j < count ? order_key[j] : 0;
    __syncthreads();
    const int m = min(kRankThreads, count - j0);
    for (int u = 0; u < m; ++u) {
      if (!s_live[u]) continue;
      ++total;
      const int32_t g = s_group[u];
      const int64_t o = s_key[u];
      rank += g < gi || (g == gi && (o < oi || (o == oi && j0 + u < i)));
    }
    __syncthreads();
  }
  if (live) {
    SOD_DCHECK(rank < count);
    for (int f = 0; f < 6; ++f) t.smean[6 * rank + f] = mean[6 * static_cast<size_t>(i) + f];
    t.sseg[rank] = gi / groups_per_frame;
  }
  if (i == 0) t.count[1] = total;
}

// Sort keys (in input order; segment_sort_kernel sorts them in place unless they are already ascending) and the
// per-bin root slots.
__global__ void pose_prep_kernel(const int32_t* __restrict__ segment, const int32_t* __restrict__ n_dev, int n,
                                 PoseTmp t) {
  const int count = n_dev ? min(max(*n_dev, 0), n) : n;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0) {
    t.count[0] = count;
    t.count[2] = 0;
    t.count[3] = 0;
  }
  if (i >= n) return;
  t.key[i] = i < count ? (segment ? segment_key(segment[i]) : segment_key(0)) : kKeyEnd;
  t.bin[i] = i;
  t.root_size[i] = 0;
}

// Stable sort of the n keys (and their bins) in key / bin by one CTA: LSD radix sort on 8-bit digits, four passes
// through key_in / bin_in and back.  Each warp owns a contiguous chunk; the counters are scanned in (digit, warp)
// order, and inside a step of 32 keys the lanes of equal digit (__match_any_sync) take consecutive slots in lane
// order, so equal keys keep their input order.  A pass whose digit is the same for every key (the high bytes of
// small segment ids) is skipped.  Needs no device query to size, unlike a library sort.
__global__ void __launch_bounds__(kSortThreads) segment_sort_kernel(PoseTmp t, int n) {
  using Scan = cub::BlockScan<int, kSortThreads>;
  __shared__ int s_base[256 * kSortWarps];          // [digit][warp]
  __shared__ typename Scan::TempStorage s_scan;
  __shared__ uint32_t s_lo, s_hi;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int chunk = (n + kSortWarps - 1) / kSortWarps;
  const int lo = min(warp * chunk, n), hi = min(lo + chunk, n);
  uint32_t *ksrc = t.key, *kdst = t.key_in;
  int32_t *bsrc = t.bin, *bdst = t.bin_in;
  constexpr int kPer = 256 * kSortWarps / kSortThreads;
  for (int shift = 0; shift < 32; shift += 8) {
    for (int i = threadIdx.x; i < 256 * kSortWarps; i += kSortThreads) s_base[i] = 0;
    if (threadIdx.x == 0) {
      s_lo = 255u;
      s_hi = 0u;
    }
    __syncthreads();
    for (int i = lo + lane; i < hi; i += 32) {
      const uint32_t d = (ksrc[i] >> shift) & 255u;
      atomicAdd(&s_base[d * kSortWarps + warp], 1);
      atomicMin(&s_lo, d);
      atomicMax(&s_hi, d);
    }
    __syncthreads();
    const bool one_digit = s_lo == s_hi;  // the pass would keep the order
    __syncthreads();                      // every thread has read s_lo / s_hi before the next pass resets them
    if (one_digit) continue;
    int v[kPer], sum = 0;
    for (int j = 0; j < kPer; ++j) sum += (v[j] = s_base[threadIdx.x * kPer + j]);
    int base;
    Scan(s_scan).ExclusiveSum(sum, base);
    for (int j = 0; j < kPer; ++j) {
      s_base[threadIdx.x * kPer + j] = base;
      base += v[j];
    }
    __syncthreads();
    for (int i0 = lo; i0 < hi; i0 += 32) {
      const int i = i0 + lane;
      const bool ok = i < hi;
      const uint32_t k = ok ? ksrc[i] : 0u;
      const int32_t b = ok ? bsrc[i] : 0;
      const int d = ok ? static_cast<int>((k >> shift) & 255u) : 256 + lane;   // idle lanes: a digit of their own
      const uint32_t peers = __match_any_sync(0xffffffffu, d);
      const int rank = __popc(peers & ((1u << lane) - 1u));
      int* slot = &s_base[(d & 255) * kSortWarps + warp];
      const int at = ok ? *slot + rank : 0;
      __syncwarp();
      if (ok) {
        SOD_DCHECK(at < n);
        kdst[at] = k;
        bdst[at] = b;
        if (rank == 0) *slot += __popc(peers);
      }
      __syncwarp();
    }
    __syncthreads();
    uint32_t* kt = ksrc; ksrc = kdst; kdst = kt;
    int32_t* bt = bsrc; bsrc = bdst; bdst = bt;
  }
  if (ksrc != t.key) {                  // an odd number of passes ran: the result is in key_in / bin_in
    for (int i = threadIdx.x; i < n; i += kSortThreads) {
      t.key[i] = ksrc[i];
      t.bin[i] = bsrc[i];
    }
  }
}

// Per sorted position: the pair-test operands (coalesced for the row kernels) and the segment's bounds.
__global__ void pose_gather_kernel(const double* __restrict__ mean, PoseTmp t) {
  const int count = t.count[0];
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= count) return;
  const int b = t.bin[q];
  const double* m = mean + 6 * static_cast<size_t>(b);
  const double s = m[3];
  t.x[q] = m[0];
  t.y[q] = m[1];
  t.ang[q] = m[2];
  t.rx[q] = pose_reach(m[4], s);
  t.ry[q] = pose_reach(m[5], s);
  const uint32_t k = t.key[q];
  int lo = 0, hi = q;              // first position of key k
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (t.key[mid] < k) lo = mid + 1; else hi = mid;
  }
  int lo2 = q + 1, hi2 = count;    // one past its last
  while (lo2 < hi2) {
    const int mid = (lo2 + hi2) >> 1;
    if (t.key[mid] <= k) lo2 = mid + 1; else hi2 = mid;
  }
  t.seg_lo[q] = lo;
  t.seg_len[q] = lo2 - lo;
  if (lo == q) t.seg_list[atomicAdd(t.count + 2, 1)] = q;
}

// group_position's bit rows: one CTA per sorted position i, row i of its segment (columns = the segment's bins).
__global__ void __launch_bounds__(kThreads) pose_rows_kernel(PoseTmp t) {
  const int i = blockIdx.x;
  if (i >= t.count[0]) return;
  const int lo = t.seg_lo[i], v = t.seg_len[i], words = (v + 31) >> 5;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const double xi = t.x[i], yi = t.y[i], rxi = t.rx[i], ryi = t.ry[i];
  uint32_t* row = t.adj + lo * t.words_cap + static_cast<int64_t>(i - lo) * words;
  for (int w = warp; w < words; w += kThreads / 32) {
    const int j = lo + w * 32 + lane;
    const bool edge = j < lo + v && j != i && position_edge(xi, yi, rxi, ryi, t.x[j], t.y[j], t.rx[j], t.ry[j]);
    const uint32_t word = __ballot_sync(0xffffffffu, edge);
    if (lane == 0) row[w] = word;
  }
}

// group_orientation's bit rows of the clusters of more than kSmall bins: one CTA per visiting position k, row
// k - lo of its cluster (nodes = positions in the cluster's visiting order).
__global__ void __launch_bounds__(kThreads) orientation_rows_kernel(PoseTmp t) {
  const int k = blockIdx.x;
  if (k >= t.count[0]) return;
  const int lo = t.cl_lo[k], m = t.cl_len[k], words = (m + 31) >> 5;
  if (m <= kSmall) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const double ak = t.oang[k];
  uint32_t* row = t.adj + lo * t.words_cap + static_cast<int64_t>(k - lo) * words;
  for (int w = warp; w < words; w += kThreads / 32) {
    const int j = lo + w * 32 + lane;
    const bool edge = j < lo + m && j != k && angle_edge(ak, t.oang[j], 1.0);
    const uint32_t word = __ballot_sync(0xffffffffu, edge);
    if (lane == 0) row[w] = word;
  }
}

// The reference's dfs (PostProcessing.py:4-11) over a graph of n nodes given as bit rows (row v at adj + v * words),
// by one warp: components from the lowest unvisited node, each step to the lowest unvisited neighbour.  The visited
// set only grows, so a node's scan resumes at the row word where it stopped (cursor[v]); each step ANDs up to 32
// words with ~visited and takes the first set bit by ballot.  visit(k, v, starts) runs on lane 0 for the k-th node
// of the walk; done(k0, m) on all lanes when a component of m nodes starting at walk position k0 is complete.
template <class Visit, class Done>
__device__ void warp_preorder(const uint32_t* __restrict__ adj, int n, uint32_t* vis, int32_t* cursor,
                              int32_t* stack, Visit visit, Done done) {
  const int lane = threadIdx.x & 31;
  const int words = (n + 31) >> 5;
  for (int w = lane; w < words; w += 32) vis[w] = 0u;
  __syncwarp();
  int k = 0;
  for (int s = 0; s < n; ++s) {
    if ((vis[s >> 5] >> (s & 31)) & 1u) continue;
    const int k0 = k;
    if (lane == 0) {
      vis[s >> 5] |= 1u << (s & 31);
      cursor[s] = 0;
      stack[0] = s;
      visit(k, s, true);
    }
    ++k;
    int sp = 1, v = s;
    __syncwarp();
    for (;;) {
      int c = cursor[v], next = -1;
      for (; c < words; c += 32) {
        const int w = c + lane;
        const uint32_t x = w < words ? adj[static_cast<int64_t>(v) * words + w] & ~vis[w] : 0u;
        const uint32_t hit = __ballot_sync(0xffffffffu, x != 0u);
        if (hit) {
          const int l = __ffs(hit) - 1;
          const uint32_t xw = __shfl_sync(0xffffffffu, x, l);
          c += l;
          next = c * 32 + __ffs(xw) - 1;
          break;
        }
      }
      if (next >= 0) {
        SOD_DCHECK(next < n && sp < n);
        if (lane == 0) {
          cursor[v] = c;
          vis[next >> 5] |= 1u << (next & 31);
          cursor[next] = 0;
          stack[sp] = next;
          visit(k, next, false);
        }
        ++sp;
        ++k;
        v = next;
      } else {
        if (--sp == 0) break;
        v = stack[sp - 1];
      }
      __syncwarp();
    }
    done(k0, k - k0);
    __syncwarp();
  }
}

// The same walk for a graph of m <= 32 nodes whose rows are held by the lanes (lane p: row p).
template <class Visit>
__device__ void warp_preorder_small(uint32_t row, int m, Visit visit) {
  const int lane = threadIdx.x & 31;
  uint32_t vis = 0u;
  int stk = 0, k = 0;               // stack entry sp lives in lane sp
  for (int s = 0; s < m; ++s) {
    if ((vis >> s) & 1u) continue;
    vis |= 1u << s;
    visit(k++, s, true);
    if (lane == 0) stk = s;
    int sp = 1, v = s;
    for (;;) {
      const uint32_t cand = __shfl_sync(0xffffffffu, row, v) & ~vis;
      if (cand) {
        const int nb = __ffs(cand) - 1;
        vis |= 1u << nb;
        visit(k++, nb, false);
        if (lane == sp) stk = nb;
        ++sp;
        v = nb;
      } else {
        if (--sp == 0) break;
        v = __shfl_sync(0xffffffffu, stk, sp - 1);
      }
    }
  }
}

// group_position's walk: one warp per segment (CTA b takes segments b, b + grid, ... of the start list).  Visiting
// position k of a segment starting at lo is lo + k; its cluster's first position and size go to cl_lo / cl_len, and
// the cluster's first position to the cluster list.
__global__ void __launch_bounds__(32) position_walk_kernel(PoseTmp t) {
  __shared__ uint32_t s_vis[kVisWords];
  const int lane = threadIdx.x;
  const int segments = t.count[2];
  SOD_DCHECK(segments <= t.count[0]);
  for (int s = blockIdx.x; s < segments; s += gridDim.x) {
    const int lo = t.seg_list[s];
    const int v = t.seg_len[lo];
    const uint32_t* adj = t.adj + lo * t.words_cap;
    warp_preorder(
        adj, v, s_vis, t.cursor + lo, t.stack + lo,
        [&](int k, int node, bool) {
          t.order[lo + k] = lo + node;
          t.oang[lo + k] = t.ang[lo + node];
        },
        [&](int k0, int m) {
          if (lane == 0) t.cl_list[atomicAdd(t.count + 3, 1)] = lo + k0;
          for (int k = lane; k < m; k += 32) {
            t.cl_lo[lo + k0 + k] = lo + k0;
            t.cl_len[lo + k0 + k] = m;
          }
        });
  }
}

// find_max_orientation and get_final_pose of one cluster (visiting positions lo..lo+m), by one thread, every
// fp64 operation rounded on its own: the reference's sequential sums in visiting order.
__device__ void cluster_pose(const double* __restrict__ mean, const PoseTmp& t, int lo, int m) {
  int best = 0;
  double ori = 0.0;
  for (int k = 0; k < m;) {           // the largest sub-cluster, later ones win ties (PostProcessing.py:65-82)
    int e = k + 1;
    while (e < m && !t.sub_first[lo + e]) ++e;
    if (e - k >= best) {
      best = e - k;
      double s = 0.0;
      for (int u = k; u < e; ++u) s = __dadd_rn(s, t.ang[t.sub[lo + u]]);
      ori = __ddiv_rn(s, static_cast<double>(e - k));
    }
    k = e;
  }
  double sx = 0.0, sy = 0.0, ss = 0.0, min_area = __longlong_as_double(0x7ff0000000000000ll);
  int shape = -1;
  for (int k = 0; k < m; ++k) {       // PostProcessing.py:86-112
    const int b = t.bin[t.order[lo + k]];
    const double* p = mean + 6 * static_cast<size_t>(b);
    const double s = p[3];
    sx = __dadd_rn(sx, p[0]);
    sy = __dadd_rn(sy, p[1]);
    ss = __dadd_rn(ss, s);
    const double area = __dmul_rn(__dmul_rn(p[4], s), __dmul_rn(p[5], s));
    if (area < min_area) {
      min_area = area;
      shape = b;
    }
  }
  const int root = t.bin[t.order[lo]];
  const double cnt = static_cast<double>(m);
  double* out = t.root_pose + 6 * static_cast<size_t>(root);
  out[0] = __ddiv_rn(sx, cnt);
  out[1] = __ddiv_rn(sy, cnt);
  out[2] = ori;
  out[3] = __ddiv_rn(ss, cnt);
  out[4] = shape >= 0 ? mean[6 * static_cast<size_t>(shape) + 4] : 0.0;
  out[5] = shape >= 0 ? mean[6 * static_cast<size_t>(shape) + 5] : 0.0;
  t.root_shape[root] = shape;
  t.root_k[root] = lo;
  t.root_size[root] = m;
}

// group_orientation's walk and the sums: one warp per cluster (CTA b takes clusters b, b + grid, ... of the list).
// sub[k] is the sorted position of the k-th node of the sub-cluster walk, sub_first[k] = 1 where one starts.
__global__ void __launch_bounds__(32) orientation_walk_kernel(const double* __restrict__ mean, PoseTmp t) {
  __shared__ uint32_t s_vis[kVisWords];
  const int lane = threadIdx.x;
  const int clusters = t.count[3];
  SOD_DCHECK(clusters <= t.count[0]);
  for (int c = blockIdx.x; c < clusters; c += gridDim.x) {
    const int lo = t.cl_list[c];
    const int m = t.cl_len[lo];
    auto visit = [&](int k, int p, bool first) {
      t.sub[lo + k] = t.order[lo + p];
      t.sub_first[lo + k] = first;
    };
    if (m <= kSmall) {
      const double a = lane < m ? t.oang[lo + lane] : 0.0;
      uint32_t row = 0u;
      for (int p = 0; p < m; ++p) {
        const double ap = __shfl_sync(0xffffffffu, a, p);
        const uint32_t r = __ballot_sync(0xffffffffu, lane < m && lane != p && angle_edge(ap, a, 1.0));
        if (lane == p) row = r;
      }
      warp_preorder_small(row, m, [&](int k, int p, bool first) {
        if (lane == 0) visit(k, p, first);
      });
    } else {
      warp_preorder(t.adj + lo * t.words_cap, m, s_vis, t.cursor + lo, t.stack + lo, visit, [](int, int) {});
    }
    __syncwarp();
    if (lane == 0) cluster_pose(mean, t, lo, m);
    __syncwarp();
  }
}

// Clusters numbered by their lowest bin (an exclusive scan over the bins of (is lowest bin, cluster size)), then
// every visiting position scattered to its cluster's output range.
__global__ void __launch_bounds__(kFinishThreads) pose_finish_kernel(PoseTmp t, sod_poses_out out) {
  using Scan = cub::BlockScan<long long, kFinishThreads>;
  __shared__ typename Scan::TempStorage s_scan;
  const int count = t.count[0];
  const int chunk = (count + kFinishThreads - 1) / kFinishThreads;
  const int b0 = min(threadIdx.x * chunk, count), b1 = min(b0 + chunk, count);
  long long mine = 0;
  for (int b = b0; b < b1; ++b) {
    const int m = t.root_size[b];
    if (m) mine += (1ll << 32) + m;
  }
  long long base, total;
  Scan(s_scan).ExclusiveSum(mine, base, total);
  int c = static_cast<int>(base >> 32), off = static_cast<int>(base & 0xffffffffll);
  for (int b = b0; b < b1; ++b) {
    const int m = t.root_size[b];
    if (!m) continue;
    SOD_DCHECK(c < count && off + m <= count);
    t.root_dst[b] = off;
    out.cluster_offset[c] = off;
    for (int f = 0; f < 6; ++f) out.pose[6 * static_cast<size_t>(c) + f] = t.root_pose[6 * static_cast<size_t>(b) + f];
    out.shape_bin[c] = t.root_shape[b];
    out.segment[c] = static_cast<int32_t>(t.key[t.root_k[b]] ^ 0x80000000u);
    ++c;
    off += m;
  }
  if (threadIdx.x == 0) {
    const int clusters = static_cast<int>(total >> 32);
    out.counters[0] = clusters;
    out.counters[1] = count;
    out.cluster_offset[clusters] = count;
  }
  __syncthreads();
  for (int k = threadIdx.x; k < count; k += kFinishThreads) {
    const int lo = t.cl_lo[k];
    const int root = t.bin[t.order[lo]];
    const int d = t.root_dst[root] + (k - lo);
    SOD_DCHECK(d >= 0 && d < count);
    out.cluster_bins[d] = t.bin[t.order[k]];
    out.sub_bins[d] = t.bin[t.sub[k]];
    out.sub_first[d] = t.sub_first[k];
  }
}

int check_poses_out(const sod_poses_out* out, int64_t n) {
  SOD_CHECK_ARG(out, "null pointer: out");
  SOD_CHECK_ARG(out->counters && out->cluster_bins && out->cluster_offset && out->sub_bins && out->sub_first &&
                    out->pose && out->shape_bin && out->segment,
                "null pointer in out");
  SOD_CHECK_ARG(out->cap >= n, "out->cap %lld < %lld bins", (long long)out->cap, (long long)n);
  return SOD_OK;
}

// Everything after the sort keys: clusters of the first count bins of mean (sorted by segment first unless
// presorted or unsegmented).
int run_final_poses(const double* mean, const int32_t* segment, int64_t n, const int32_t* n_dev, int presorted,
                    const sod_poses_out* out, void* workspace, cudaStream_t st) {
  PoseTmp t = pose_tmp(workspace, n);
  const int ni = static_cast<int>(n);
  const unsigned blocks = static_cast<unsigned>((ni + kThreads - 1) / kThreads);
  pose_prep_kernel<<<blocks, kThreads, 0, st>>>(segment, n_dev, ni, t);
  SOD_CHECK_LAUNCH("pose_prep_kernel");
  if (segment && !presorted) {
    segment_sort_kernel<<<1, kSortThreads, 0, st>>>(t, ni);
    SOD_CHECK_LAUNCH("segment_sort_kernel");
  }
  pose_gather_kernel<<<blocks, kThreads, 0, st>>>(mean, t);
  SOD_CHECK_LAUNCH("pose_gather_kernel");
  pose_rows_kernel<<<static_cast<unsigned>(ni), kThreads, 0, st>>>(t);
  SOD_CHECK_LAUNCH("pose_rows_kernel");
  const unsigned walks = static_cast<unsigned>(ni < kWalkGrid ? ni : kWalkGrid);
  position_walk_kernel<<<walks, 32, 0, st>>>(t);
  SOD_CHECK_LAUNCH("position_walk_kernel");
  orientation_rows_kernel<<<static_cast<unsigned>(ni), kThreads, 0, st>>>(t);
  SOD_CHECK_LAUNCH("orientation_rows_kernel");
  orientation_walk_kernel<<<walks, 32, 0, st>>>(mean, t);
  SOD_CHECK_LAUNCH("orientation_walk_kernel");
  pose_finish_kernel<<<1, kFinishThreads, 0, st>>>(t, *out);
  SOD_CHECK_LAUNCH("pose_finish_kernel");
  return SOD_OK;
}

}  // namespace
}  // namespace sod

using namespace sod;

extern "C" {

int sod_pose_adjacency(const double* cx, const double* cy, const double* reach_x, const double* reach_y,
                       const int32_t* segment, int64_t n, uint32_t* adj, int32_t* label, sod_stream_t stream) {
  return run_adjacency<0>(cx, cy, reach_x, reach_y, segment, n, 0.0, adj, label, stream);
}

int sod_angle_adjacency(const double* angle, const int32_t* segment, int64_t n, double max_degrees, uint32_t* adj,
                        int32_t* label, sod_stream_t stream) {
  return run_adjacency<1>(angle, nullptr, nullptr, nullptr, segment, n, max_degrees, adj, label, stream);
}

size_t sod_final_poses_workspace_bytes(int64_t cap) {
  if (cap < 0 || cap > SOD_MAX_CLUSTER_BINS) return 0;
  return pose_layout(cap).total;
}

int sod_final_poses(const double* mean, const int32_t* segment, int64_t n, const int32_t* n_dev,
                    const sod_poses_out* out, void* workspace, size_t workspace_bytes, sod_stream_t stream) {
  SOD_CHECK_ARG(n >= 0 && n <= SOD_MAX_CLUSTER_BINS, "n must be in 0..%d", SOD_MAX_CLUSTER_BINS);
  if (n == 0) return SOD_OK;
  SOD_CHECK_ARG(mean && workspace, "null pointer");
  const int rc = check_poses_out(out, n);
  if (rc != SOD_OK) return rc;
  SOD_CHECK_ARG(workspace_bytes >= pose_layout(n).total, "workspace too small: %zu < %zu bytes", workspace_bytes,
                pose_layout(n).total);
  return run_final_poses(mean, segment, n, n_dev, 0, out, workspace, static_cast<cudaStream_t>(stream));
}

int sod_final_poses_records(const int32_t* status, const int32_t* group, const int64_t* order_key,
                            const double* mean, int64_t cap, const int32_t* n_dev, int32_t groups_per_frame,
                            const sod_poses_out* out, void* workspace, size_t workspace_bytes,
                            sod_stream_t stream) {
  SOD_CHECK_ARG(cap >= 0 && cap <= SOD_MAX_CLUSTER_BINS, "cap must be in 0..%d", SOD_MAX_CLUSTER_BINS);
  SOD_CHECK_ARG(groups_per_frame >= 1, "groups_per_frame must be >= 1");
  if (cap == 0) return SOD_OK;
  SOD_CHECK_ARG(status && group && order_key && mean && n_dev && workspace, "null pointer");
  const int rc = check_poses_out(out, cap);
  if (rc != SOD_OK) return rc;
  SOD_CHECK_ARG(workspace_bytes >= pose_layout(cap).total, "workspace too small: %zu < %zu bytes", workspace_bytes,
                pose_layout(cap).total);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  PoseTmp t = pose_tmp(workspace, cap);
  const int ci = static_cast<int>(cap);
  live_rank_kernel<<<static_cast<unsigned>((ci + kRankThreads - 1) / kRankThreads), kRankThreads, 0, st>>>(
      status, group, order_key, mean, n_dev, ci, groups_per_frame, t);
  SOD_CHECK_LAUNCH("live_rank_kernel");
  return run_final_poses(t.smean, t.sseg, cap, t.count + 1, 1, out, workspace, st);
}

}  // extern "C"
