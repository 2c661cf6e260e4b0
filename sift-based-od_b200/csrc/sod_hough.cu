// K4: generalized Hough voting (pose estimate, bin index, 16 votes per match, PoseBin bookkeeping)
// and the stable compaction of ratio survivors that feeds it.
//
// Replaces Main.apply_hough_transform (main.py:89-119), estimate_object_pose / calculate_bin_index
// (HoughTransformHelperFunctions.py:4-72), unpack_sift_octave (SiftHelperFunctions.py:25-40) and
// PoseBin.update_posebin (PoseBin.py:19-54).
//
// Data flow (all on the caller's stream, no host synchronisation):
//   pose    one thread per match: fp64 pose with the reference's operation order (explicit
//           round-to-nearest intrinsics, no FMA contraction), base bin, Hough-space (group) id
//   group   counting sort of the matches by group
//   vote    one CTA per group at a time: a bins^4 uint32 histogram privatised in shared memory
//           (202.5 KB at bins = 15) takes the <=16 votes of every match with shared-memory atomics;
//           the vote that finds a zero counter owns ("creates") the bin and later emits its compact
//           record, so the cost is proportional to the votes, not to the 50,625 bins
//   finish  one warp per bin record: members sorted by match id (= reference append order), running
//           means by the reference's sequential recurrence, insertion-order key
#include <climits>

#include "sod_common.cuh"

namespace sod {
namespace {

constexpr double kTwoPi = 2.0 * 3.141592653589793;  // 2*math.pi (exact doubling)
constexpr double kDegToRad = 3.141592653589793 / 180.0;  // CPython's math.radians multiplier
constexpr int kVoteThreads = 1024;
constexpr int kGroupChunk = 256;  // most Hough spaces examined per work-stealing ticket

__device__ __forceinline__ int sext8(int v) {
  const int o = v & 0xFF;
  return o >= 128 ? o - 256 : o;
}

// Near a truncation boundary?  cos/sin on the device may differ from the host libm in the last
// bits; only values this close to an integer could then land in another bin.
__device__ __forceinline__ bool near_integer(double f) {
  const double r = rint(f);
  return fabs(f - r) <= 1e-9 * fmax(1.0, fabs(f));
}

// v moved by `ulps` units in the last place, away from (ulps > 0) or towards (ulps < 0) zero.
__device__ __forceinline__ double step_ulps(double v, int ulps) {
  return __longlong_as_double(__double_as_longlong(v) + ulps);
}

// x, y of estimate_object_pose and their truncated bin coordinates for given cos / sin values, in the
// reference's operation order (HoughTransformHelperFunctions.py:28-32, 49-57).
struct XyBins {
  double x, y, fx, fy;
  int tx, ty;  // int(x*bins/W), int(y*bins/H) before the -1 shift and the clamp
};
__device__ __forceinline__ XyBins xy_bins(double ca, double sa, double tx, double ty, double qx, double qy,
                                          double bx, double by, double W, double H) {
  XyBins r;
  const double rx = __dsub_rn(__dmul_rn(ca, tx), __dmul_rn(sa, ty));
  const double ry = __dadd_rn(__dmul_rn(sa, tx), __dmul_rn(ca, ty));
  r.x = __dadd_rn(rx, qx);
  r.y = __dadd_rn(ry, qy);
  r.fx = __ddiv_rn(__dmul_rn(r.x, bx), W);
  r.fy = __ddiv_rn(__dmul_rn(r.y, by), H);
  // int() truncates toward zero; clamp before converting so huge poses stay defined
  r.tx = static_cast<int>(fmin(fmax(trunc(r.fx), -1.0e6), 1.0e6));
  r.ty = static_cast<int>(fmin(fmax(trunc(r.fy), -1.0e6), 1.0e6));
  return r;
}

// Bin counts of the four pose dimensions (x, y, theta, log2 scale).  The live path uses one count
// for all four (main.py:89); the legacy perform_hough_transform takes them separately
// (HoughTransform.py:8).  A bin code is ((cx * y + cy) * t + ct) * s + cs.
struct Bins4 {
  int x, y, t, s;
  __host__ __device__ int total() const { return x * y * t * s; }
  __host__ __device__ int code(int cx, int cy, int ct, int cs) const { return ((cx * y + cy) * t + ct) * s + cs; }
};

struct PoseArgs {
  sod_scene sc;
  const int32_t* match_q;
  const int32_t* match_t;
  const int32_t* n_dev;
  int64_t n_cap;
  Bins4 bins;
  const int32_t* sigma_lut;
  double* pose;
  uint32_t* base_bin;
  uint8_t* near_edge;
  int32_t* counters;
  int32_t* group_of;
  int32_t* group_count;
  int32_t* group_rank;  // [M] arrival rank of the match inside its sub-list (the counting sort's position)
  int group_shift;      // log2 of the sub-counters per Hough space (group_sub_shift)
  double* match_size;  // [M][2] (w, h) of the match's model image, or nullptr: read again by the finish kernels
};

__device__ __forceinline__ int64_t live_count(const int32_t* n_dev, int64_t cap) {
  if (!n_dev) return cap;
  const int64_t n = *n_dev;
  return n < cap ? n : cap;
}

__global__ void hough_pose_kernel(const PoseArgs a) {
  const int64_t n = live_count(a.n_dev, a.n_cap);
  const Bins4 bins = a.bins;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int qi = a.match_q[i], ti = a.match_t[i];
    SOD_DCHECK(qi >= 0 && qi < a.sc.query.n && ti >= 0 && ti < a.sc.model.n);
    const float2 qp = reinterpret_cast<const float2*>(a.sc.query.xy)[qi];
    const float2 mp = reinterpret_cast<const float2*>(a.sc.model.xy)[ti];
    const int frame = a.sc.query_frame ? a.sc.query_frame[qi] : 0;
    const double W = a.sc.frame_wh[2 * frame], H = a.sc.frame_wh[2 * frame + 1];
    const int img = a.sc.model_image[ti];
    SOD_DCHECK(frame >= 0 && frame < a.sc.n_frames && img >= 0 && img < a.sc.n_images);
    const int grp = frame * a.sc.groups_per_frame + (a.sc.image_group ? a.sc.image_group[img] : 0);
    SOD_DCHECK(grp >= 0 && grp < a.sc.n_frames * a.sc.groups_per_frame);
    const double cx = a.sc.image_centroid[2 * img], cy = a.sc.image_centroid[2 * img + 1];
    // scale_factor = m_scale / q_scale = 2^(q_octave - m_octave), exact
    const int k = sext8(a.sc.query.octave[qi]) - sext8(a.sc.model.octave[ti]);
    const double s = ldexp(1.0, k);
    const double tx = __dmul_rn(__dsub_rn(cx, static_cast<double>(mp.x)), s);
    const double ty = __dmul_rn(__dsub_rn(cy, static_cast<double>(mp.y)), s);
    double al = __dmul_rn(__dsub_rn(static_cast<double>(a.sc.query.angle[qi]),
                                    static_cast<double>(a.sc.model.angle[ti])), kDegToRad);
    al = fmod(__dadd_rn(al, kTwoPi), kTwoPi);  // operand is > 0: Python's % equals fmod here
    if (al < 0.0) al = __dadd_rn(al, kTwoPi);
    double sa, ca;
    sincos(al, &sa, &ca);
    const double qx = static_cast<double>(qp.x), qy = static_cast<double>(qp.y);
    const double bx = static_cast<double>(bins.x), by = static_cast<double>(bins.y);
    const XyBins c = xy_bins(ca, sa, tx, ty, qx, qy, bx, by, W, H);
    double* po = a.pose + i * 4;
    po[0] = c.x; po[1] = c.y; po[2] = al; po[3] = s;
    if (a.match_size)
      reinterpret_cast<double2*>(a.match_size)[i] = reinterpret_cast<const double2*>(a.sc.image_size)[img];

    // theta and sigma bins depend on exact IEEE operations only (no libm): always bit-identical
    const double ft = fmod(__ddiv_rn(__dmul_rn(al, static_cast<double>(bins.t)), kTwoPi),
                           static_cast<double>(bins.t));
    const int ix = min(max(0, c.tx - 1), bins.x - 1);
    const int iy = min(max(0, c.ty - 1), bins.y - 1);
    const int it = static_cast<int>(ft);
    const int kk = min(max(k, SOD_SIGMA_LUT_MIN), SOD_SIGMA_LUT_MIN + SOD_SIGMA_LUT_LEN - 1);
    const int is = a.sigma_lut[kk - SOD_SIGMA_LUT_MIN];
    a.base_bin[i] = static_cast<uint32_t>(ix) | (static_cast<uint32_t>(iy) << 8) |
                    (static_cast<uint32_t>(it) << 16) | (static_cast<uint32_t>(is) << 24);
    // x and y go through cos / sin, whose last bits may differ between the device and the host libm
    // (CUDA: <= 2 ulp, glibc: < 1 ulp).  A match whose x*bins/W or y*bins/H lies within 1e-9 of an
    // integer is RESOLVED on the spot: the truncations are re-evaluated with cos and sin moved by
    // +-4 ulp (x and y are monotone in each, so the four corners bound every admissible libm); if all
    // agree, the bin is the reference's whatever its libm returns.  al == 0 is exact everywhere
    // (cos = 1, sin = 0).  Only a disagreement is left open; it is counted in counters[4].
    int edge = (near_integer(c.fx) || near_integer(c.fy)) ? 1 : 0;
    if (edge && al != 0.0) {
      bool same = true;
#pragma unroll
      for (int corner = 0; corner < 4; ++corner) {
        const XyBins p = xy_bins(step_ulps(ca, (corner & 1) ? 4 : -4), step_ulps(sa, (corner & 2) ? 4 : -4), tx, ty,
                                 qx, qy, bx, by, W, H);
        same = same && min(max(0, p.tx - 1), bins.x - 1) == ix && min(max(0, p.ty - 1), bins.y - 1) == iy;
      }
      if (!same) edge = 2;
    }
    if (a.near_edge) a.near_edge[i] = static_cast<uint8_t>(edge);
    if (edge && a.counters) {
      atomicAdd(&a.counters[2], 1);
      if (edge == 2) atomicAdd(&a.counters[4], 1);
    }
    if (a.group_of) {
      // Position inside the Hough space = the counting atomic's return value.  Consecutive matches often
      // belong to one space (a stress scene holds thousands per object): the lanes of a warp that share a
      // space take their positions with ONE atomic (2 M same-address atomics with return were most of this
      // kernel's time at C5).  The order inside a space is free - the finish kernels sort members by match id.
      // A scene with few spaces would send all those atomics to a handful of L2 lines (500 spaces = 16 lines
      // took 2 M atomics at C5: 0.3 ms).  Each space therefore owns 2^group_shift sub-counters, picked by the
      // warp's number: the space's matches form that many sub-lists, laid out one after the other by the scan.
      const int sub = (grp << a.group_shift) +
                      (static_cast<int>(i >> 5) & ((1 << a.group_shift) - 1));  // the same for the whole warp
      a.group_of[i] = sub;
      const unsigned lane = threadIdx.x & 31u;
      const unsigned peers = __match_any_sync(__activemask(), grp);
      const int leader = __ffs(peers) - 1;
      int first = 0;
      if (static_cast<int>(lane) == leader) first = atomicAdd(&a.group_count[sub], __popc(peers));
      first = __shfl_sync(peers, first, leader);
      a.group_rank[i] = first + __popc(peers & ((1u << lane) - 1u));
    }
  }
}

// calculate_bin_index for caller-supplied poses (the drop-in helper of the same name).  The scale
// need not be a power of two here: exact powers use the table, others log(s)/log(2) on the device.
__global__ void pose_bin_index_kernel(const double* __restrict__ pose, int64_t n, int bins, double W,
                                      double H, const int32_t* __restrict__ sigma_lut,
                                      uint32_t* __restrict__ base_bin) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double x = pose[4 * i], y = pose[4 * i + 1], al = pose[4 * i + 2], s = pose[4 * i + 3];
  const double fx = __ddiv_rn(__dmul_rn(x, static_cast<double>(bins)), W);
  const double fy = __ddiv_rn(__dmul_rn(y, static_cast<double>(bins)), H);
  double ft = fmod(__ddiv_rn(__dmul_rn(al, static_cast<double>(bins)), kTwoPi), static_cast<double>(bins));
  if (ft < 0.0) ft = __dadd_rn(ft, static_cast<double>(bins));  // Python's % follows the divisor's sign
  int ix = static_cast<int>(fmin(fmax(trunc(fx), -1.0e6), 1.0e6));
  int iy = static_cast<int>(fmin(fmax(trunc(fy), -1.0e6), 1.0e6));
  ix = min(max(0, ix - 1), bins - 1);
  iy = min(max(0, iy - 1), bins - 1);
  int it = min(max(static_cast<int>(ft), 0), bins - 1);
  int e = 0;
  const double mant = frexp(s, &e);
  int is;
  if (mant == 0.5 && e - 1 >= SOD_SIGMA_LUT_MIN && e - 1 < SOD_SIGMA_LUT_MIN + SOD_SIGMA_LUT_LEN) {
    is = sigma_lut[e - 1 - SOD_SIGMA_LUT_MIN];
  } else {
    const double v = __dmul_rn(__ddiv_rn(__ddiv_rn(log(s), log(2.0)), 6.5), static_cast<double>(bins));
    is = min(max(static_cast<int>(fmin(fmax(trunc(v), -1.0e6), 1.0e6)), 0), bins - 1);
  }
  base_bin[i] = static_cast<uint32_t>(ix) | (static_cast<uint32_t>(iy) << 8) |
                (static_cast<uint32_t>(it) << 16) | (static_cast<uint32_t>(is) << 24);
}

// Inclusive prefix sum of v over the lanes of a warp.
__device__ __forceinline__ int warp_inclusive_scan(int v) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += t;
  }
  return v;
}

// Exclusive prefix sum of v over a CTA of 32 warps: the warps' totals meet in warp_sums[32] (shared memory),
// warp 0 turns them into the warps' exclusive prefixes, every thread adds its own warp's.  Every thread must
// call it.  The CTA's total is the last thread's result + v.
__device__ __forceinline__ int cta_exclusive_scan(int v, int* warp_sums) {
  SOD_DCHECK(blockDim.x == 1024);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int incl = warp_inclusive_scan(v);
  if (lane == 31) warp_sums[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    const int w = warp_sums[lane];
    warp_sums[lane] = warp_inclusive_scan(w) - w;
  }
  __syncthreads();
  return warp_sums[warp] + incl - v;
}

// Exclusive scan of n ints.  One CTA scans rounds of 8,192 elements (8 consecutive per thread) and carries
// the running total; `seed` (may be NULL) holds the value the first element starts from and `n_end` (may be
// < 0) is where the grand total is written.  Small inputs (compaction blocks) take one launch of one CTA.
// Large ones (the Hough spaces of a batch: up to a few 100k) take three: every CTA of a grid sums its own
// 8,192-element tile (scan_tile_sums_kernel), one CTA scans the tile sums, and the same kernel runs again as
// a grid with blockIdx.x selecting the tile and the scanned tile sum as its seed.
constexpr int kScanItems = 8;
constexpr int kScanTile = 1024 * kScanItems;
__global__ void __launch_bounds__(1024) exclusive_scan_kernel(const int32_t* __restrict__ in,
                                                              int64_t n, int32_t* __restrict__ out,
                                                              int32_t* __restrict__ total,
                                                              const int32_t* __restrict__ tile_seed) {
  __shared__ int32_t warp_sums[32];
  __shared__ int32_t carry;
  // grid form: this CTA owns tile blockIdx.x only and starts from the scanned sum of the tiles before it
  const int64_t first = tile_seed ? static_cast<int64_t>(blockIdx.x) * kScanTile : 0;
  const int64_t last = tile_seed ? (first + kScanTile < n ? first + kScanTile : n) : n;
  if (threadIdx.x == 0) carry = tile_seed ? tile_seed[blockIdx.x] : 0;
  __syncthreads();
  for (int64_t base = first; base < last; base += static_cast<int64_t>(blockDim.x) * kScanItems) {
    const int64_t i0 = base + static_cast<int64_t>(threadIdx.x) * kScanItems;
    int32_t v[kScanItems];
    int32_t sum = 0;
#pragma unroll
    for (int k = 0; k < kScanItems; ++k) {
      v[k] = i0 + k < n ? in[i0 + k] : 0;
      sum += v[k];
    }
    int32_t excl = carry + cta_exclusive_scan(sum, warp_sums);
#pragma unroll
    for (int k = 0; k < kScanItems; ++k) {
      if (i0 + k < n) out[i0 + k] = excl;
      excl += v[k];
    }
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) carry = excl;  // the last thread's end = the running total
    __syncthreads();
  }
  if (threadIdx.x == 0 && last == n) {
    out[n] = carry;
    if (total) *total = carry;
  }
}

__global__ void __launch_bounds__(1024) scan_tile_sums_kernel(const int32_t* __restrict__ in, int64_t n,
                                                              int32_t* __restrict__ tile_sums) {
  __shared__ int32_t warp_sums[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t i0 = static_cast<int64_t>(blockIdx.x) * kScanTile + static_cast<int64_t>(threadIdx.x) * kScanItems;
  int32_t sum = 0;
#pragma unroll
  for (int k = 0; k < kScanItems; ++k) sum += i0 + k < n ? in[i0 + k] : 0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  if (lane == 0) warp_sums[warp] = sum;
  __syncthreads();
  if (warp == 0) {
    int32_t w = warp_sums[lane];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) w += __shfl_xor_sync(0xffffffffu, w, o);
    if (lane == 0) tile_sums[blockIdx.x] = w;
  }
}

// out[0..n] = exclusive scan of in[0..n) (out[n] = total); tile_ws: 2 * (ceil(n / kScanTile) + 1) ints.
cudaError_t device_exclusive_scan(const int32_t* in, int64_t n, int32_t* out, int32_t* tile_ws, cudaStream_t st) {
  const int64_t tiles = (n + kScanTile - 1) / kScanTile;
  if (tiles <= 2 || !tile_ws) {
    exclusive_scan_kernel<<<1, 1024, 0, st>>>(in, n, out, nullptr, nullptr);
    return cudaGetLastError();
  }
  int32_t* sums = tile_ws;
  int32_t* seeds = tile_ws + tiles + 1;
  scan_tile_sums_kernel<<<static_cast<unsigned>(tiles), 1024, 0, st>>>(in, n, sums);
  exclusive_scan_kernel<<<1, 1024, 0, st>>>(sums, tiles, seeds, nullptr, nullptr);
  exclusive_scan_kernel<<<static_cast<unsigned>(tiles), 1024, 0, st>>>(in, n, out, nullptr, seeds);
  return cudaGetLastError();
}

// Counting-sort scatter: match id and its base bin travel together, so that the voting kernel reads
// both with coalesced loads instead of gathering base_bin[grouped[p]] in each of its four phases.  The
// position inside the space is the rank the pose kernel's counting atomic returned: no second atomic.
__global__ void group_scatter_kernel(const int32_t* __restrict__ group_of, const int32_t* __restrict__ group_rank,
                                     const uint32_t* __restrict__ base_bin, const int32_t* n_dev, int64_t n_cap,
                                     const int32_t* __restrict__ group_off, int32_t* __restrict__ grouped,
                                     uint32_t* __restrict__ grouped_base) {
  const int64_t n = live_count(n_dev, n_cap);
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int pos = group_off[group_of[i]] + group_rank[i];
    SOD_DCHECK(pos >= 0 && pos < n);
    grouped[pos] = static_cast<int32_t>(i);
    grouped_base[pos] = base_bin[i];
  }
}

struct VoteArgs {
  const int32_t* group_off;  // [(n_groups << group_shift) + 1]: space g = [group_off[g << shift], group_off[(g + 1) << shift])
  int group_shift;
  const int32_t* grouped;    // match ids grouped by Hough space
  const uint32_t* base_bin;  // base bins in the same (grouped) order
  uint32_t* rank;            // per grouped position 16 slots: arrival rank of each of its votes in its bin
  uint16_t* creator;         // per grouped position: which of the 16 votes created (took rank 0 of) its bin
  int64_t n_groups;
  Bins4 bins;
  int group_chunk;           // Hough spaces per ticket: 1 for few large spaces ... kGroupChunk for many sparse ones
  int32_t* ticket;           // work-stealing counter over chunks of group_chunk Hough spaces (zeroed per call)
  int32_t* counters;
  int32_t* bin_group;
  int32_t* bin_code;
  int32_t* bin_count;
  int32_t* bin_offset;
  int32_t* members_raw;
  int64_t cap_bins, cap_votes;
};

// Calls f(o, code) for each of the <=16 in-range votes of a match (main.py:105-110).
template <class F>
__device__ __forceinline__ void for_each_vote(uint32_t base, const Bins4& bins, F&& f) {
  const int ix = base & 0xFF, iy = (base >> 8) & 0xFF, it = (base >> 16) & 0xFF, is = base >> 24;
#pragma unroll
  for (int o = 0; o < 16; ++o) {
    const int cx = ix + ((o >> 3) & 1), cy = iy + ((o >> 2) & 1), ct = it + ((o >> 1) & 1),
              cs = is + (o & 1);
    if (cx < bins.x && cy < bins.y && ct < bins.t && cs < bins.s) f(o, bins.code(cx, cy, ct, cs));
  }
}

// The steps both forms of a space's vote share.  s_counts: [0] n_bins, [1] n_votes, [2] rec_base,
// [3] vote_base, [4] rec_cur, [5] vote_cur, [6] ok.
//
// After phase A: the CTA's bins and votes (each thread's my_bins / my_votes) reserve one range of records and
// one of members.  False (and counters[3] set) if either would pass its capacity.
__device__ __forceinline__ bool reserve_space(const VoteArgs& a, int my_bins, int my_votes, int* s_counts) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    my_bins += __shfl_xor_sync(0xffffffffu, my_bins, o);
    my_votes += __shfl_xor_sync(0xffffffffu, my_votes, o);
  }
  if ((threadIdx.x & 31) == 0 && my_votes) {
    atomicAdd(&s_counts[0], my_bins);
    atomicAdd(&s_counts[1], my_votes);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    s_counts[2] = atomicAdd(&a.counters[0], s_counts[0]);
    s_counts[3] = atomicAdd(&a.counters[1], s_counts[1]);
    s_counts[6] = (static_cast<int64_t>(s_counts[2]) + s_counts[0] <= a.cap_bins) &&
                  (static_cast<int64_t>(s_counts[3]) + s_counts[1] <= a.cap_votes);
    if (!s_counts[6]) a.counters[3] = 1;
  }
  __syncthreads();
  return s_counts[6] != 0;
}

// Phase B for one match: each vote that created its bin emits the bin record and turns the bin's counter
// into the offset of its members.
__device__ __forceinline__ void emit_created_bins(const VoteArgs& a, uint32_t* hist, int64_t g, uint32_t base,
                                                  const Bins4& bins, unsigned created, const int& rec_base,
                                                  const int& vote_base, int* s_counts) {
  for_each_vote(base, bins, [&](int o, int code) {
    if (!(created >> o & 1u)) return;
    const int cnt = static_cast<int>(hist[code]);
    const int rec = rec_base + atomicAdd(&s_counts[4], 1);
    const int off = vote_base + atomicAdd(&s_counts[5], cnt);
    SOD_DCHECK(rec < a.cap_bins && static_cast<int64_t>(off) + cnt <= a.cap_votes);
    a.bin_group[rec] = static_cast<int32_t>(g);
    a.bin_code[rec] = code;
    a.bin_count[rec] = cnt;
    a.bin_offset[rec] = off;
    hist[code] = static_cast<uint32_t>(off);
  });
}

// Phase C for one vote: match m at the bin's offset + the vote's arrival rank r.
__device__ __forceinline__ void store_member(const VoteArgs& a, const uint32_t* hist, int code, uint32_t r, int m) {
  SOD_DCHECK(static_cast<int64_t>(hist[code]) + r < a.cap_votes);
  a.members_raw[hist[code] + r] = m;
}

// Phase D for one match: the bins it created get their counters back to zero.
__device__ __forceinline__ void clear_created_bins(uint32_t* hist, uint32_t base, const Bins4& bins, unsigned created) {
  for_each_vote(base, bins, [&](int o, int code) {
    if (created >> o & 1u) hist[code] = 0u;
  });
}

// One Hough space: the four phases over the matches [beg, end) of the space.  kWide: arrival ranks as
// 32-bit values (spaces of more than 65,535 matches), else packed 16-bit pairs (half the traffic).
//  A  every vote takes the next rank of its bin: ONE shared-memory atomic per vote; rank 0 created the bin.
//     The 16 ranks of a match stay in registers and leave as two (four) 16-byte stores, the creator bits
//     as one 16-bit mask.
//  B  the creating vote emits the bin record and turns the counter into the bin's offset
//  C  every vote stores its match id at offset + rank: no atomic, the ranks of phase A are a permutation
//  D  creators clear their counters for the next space
template <bool kWide>
__device__ __forceinline__ void vote_space(const VoteArgs& a, uint32_t* hist, int64_t g, int beg, int end,
                                           int* s_counts) {
  constexpr int kWords = kWide ? 16 : 8;  // 32-bit words of rank storage per match
  const Bins4 bins = a.bins;
  const int tid = threadIdx.x;
  if (tid == 0) s_counts[0] = s_counts[1] = s_counts[4] = s_counts[5] = 0;
  __syncthreads();
  int my_bins = 0, my_votes = 0;
  for (int p = beg + tid; p < end; p += kVoteThreads) {
    uint32_t rk[kWords];
#pragma unroll
    for (int i = 0; i < kWords; ++i) rk[i] = 0u;
    unsigned created = 0;
    for_each_vote(a.base_bin[p], bins, [&](int o, int code) {
      SOD_DCHECK(code >= 0 && code < bins.total());
      const uint32_t r = atomicAdd(&hist[code], 1u);
      SOD_DCHECK(kWide || r <= 0xFFFFu);
      if (kWide) rk[o] = r;
      else rk[o >> 1] |= r << ((o & 1) * 16);
      created |= (r == 0u ? 1u : 0u) << o;
      ++my_votes;
    });
    uint4* dst = reinterpret_cast<uint4*>(a.rank + static_cast<int64_t>(p) * 16);
#pragma unroll
    for (int i = 0; i < kWords / 4; ++i) dst[i] = make_uint4(rk[4 * i], rk[4 * i + 1], rk[4 * i + 2], rk[4 * i + 3]);
    a.creator[p] = static_cast<uint16_t>(created);
    my_bins += __popc(created);
  }
  const bool ok = reserve_space(a, my_bins, my_votes, s_counts);
  const int rec_base = s_counts[2], vote_base = s_counts[3];
  if (ok) {
    for (int p = beg + tid; p < end; p += kVoteThreads) {
      const unsigned created = a.creator[p];
      if (!created) continue;
      emit_created_bins(a, hist, g, a.base_bin[p], bins, created, rec_base, vote_base, s_counts);
    }
  }
  __syncthreads();
  if (ok) {
    for (int p = beg + tid; p < end; p += kVoteThreads) {
      const int m = a.grouped[p];
      const uint4* src = reinterpret_cast<const uint4*>(a.rank + static_cast<int64_t>(p) * 16);
      uint32_t rk[kWords];
#pragma unroll
      for (int i = 0; i < kWords / 4; ++i) {
        const uint4 v = src[i];
        rk[4 * i] = v.x; rk[4 * i + 1] = v.y; rk[4 * i + 2] = v.z; rk[4 * i + 3] = v.w;
      }
      for_each_vote(a.base_bin[p], bins, [&](int o, int code) {
        store_member(a, hist, code, kWide ? rk[o] : (rk[o >> 1] >> ((o & 1) * 16)) & 0xFFFFu, m);
      });
    }
  }
  __syncthreads();
  for (int p = beg + tid; p < end; p += kVoteThreads) {
    const unsigned created = a.creator[p];
    if (!created) continue;
    clear_created_bins(hist, a.base_bin[p], bins, created);
  }
  __syncthreads();
}

// The same four phases for a space of at most kVoteThreads matches (every space of the bench workload: a
// (frame, object) pair holds a handful): one match per thread, so its base bin, ranks, creator bits and match
// id stay in REGISTERS from phase to phase - the general form's stores and re-loads of a.rank / a.creator /
// a.base_bin are dependent global round trips, which is most of what a small space costs.
__device__ __forceinline__ void vote_space_small(const VoteArgs& a, uint32_t* hist, int64_t g, int beg, int end,
                                                 int* s_counts) {
  const Bins4 bins = a.bins;
  const int tid = threadIdx.x;
  const int p = beg + tid;
  const bool have = p < end;
  if (tid == 0) s_counts[0] = s_counts[1] = s_counts[4] = s_counts[5] = 0;
  __syncthreads();
  uint32_t base = 0, rk[8];
  int m = 0, my_votes = 0;
  unsigned created = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) rk[i] = 0u;
  if (have) {
    base = a.base_bin[p];
    m = a.grouped[p];
    for_each_vote(base, bins, [&](int o, int code) {
      SOD_DCHECK(code >= 0 && code < bins.total());
      const uint32_t r = atomicAdd(&hist[code], 1u);  // r < kVoteThreads: 16 bits hold it
      rk[o >> 1] |= r << ((o & 1) * 16);
      created |= (r == 0u ? 1u : 0u) << o;
      ++my_votes;
    });
  }
  const bool ok = reserve_space(a, __popc(created), my_votes, s_counts);
  const int rec_base = s_counts[2], vote_base = s_counts[3];
  if (ok && created) emit_created_bins(a, hist, g, base, bins, created, rec_base, vote_base, s_counts);
  __syncthreads();
  if (ok && have) {
    for_each_vote(base, bins, [&](int o, int code) {
      store_member(a, hist, code, (rk[o >> 1] >> ((o & 1) * 16)) & 0xFFFFu, m);
    });
  }
  __syncthreads();
  if (created) clear_created_bins(hist, base, bins, created);
  __syncthreads();
}

__global__ void __launch_bounds__(kVoteThreads, 1) hough_vote_kernel(const VoteArgs a) {
  extern __shared__ uint32_t hist[];  // bins^4 counters, all zero between groups
  __shared__ int s_counts[8];
  const int nb4 = a.bins.total();
  const int tid = threadIdx.x;
  __shared__ int s_chunk, s_nlist;
  __shared__ int s_list[kGroupChunk];
  for (int i = tid; i < nb4; i += kVoteThreads) hist[i] = 0;
  __syncthreads();
  // Most (frame, object) spaces are empty: CTAs steal chunks of kGroupChunk spaces, test them in
  // parallel and only walk the non-empty ones.
  for (;;) {
    if (tid == 0) {
      s_chunk = atomicAdd(a.ticket, 1);
      s_nlist = 0;
    }
    __syncthreads();
    const int64_t gbase = static_cast<int64_t>(s_chunk) * a.group_chunk;
    if (gbase >= a.n_groups) break;
    if (tid < a.group_chunk && gbase + tid < a.n_groups &&
        a.group_off[(gbase + tid + 1) << a.group_shift] > a.group_off[(gbase + tid) << a.group_shift])
      s_list[atomicAdd(&s_nlist, 1)] = tid;
    __syncthreads();
    const int n_list = s_nlist;
    for (int li = 0; li < n_list; ++li) {
      const int64_t g = gbase + s_list[li];
      const int beg = a.group_off[g << a.group_shift], end = a.group_off[(g + 1) << a.group_shift];
      if (end - beg <= kVoteThreads)
        vote_space_small(a, hist, g, beg, end, s_counts);
      else if (end - beg <= 65535)
        vote_space<false>(a, hist, g, beg, end, s_counts);
      else
        vote_space<true>(a, hist, g, beg, end, s_counts);
    }
    __syncthreads();  // s_list / s_chunk are rewritten by the next ticket
  }
}

struct FinishArgs {
  const double* pose;        // [M][4]
  const double* match_size;  // [M][2] model image size of every match (written by hough_pose_kernel)
  const uint32_t* base_bin;
  const int32_t* counters;
  const int32_t* bin_code;
  const int32_t* bin_count;
  const int32_t* bin_offset;
  const int32_t* members_raw;
  int32_t* members;
  int64_t* bin_order;
  double* bin_mean;
  int64_t cap_bins;
  Bins4 bins;
  int detail_min_count;  // bins with fewer votes get no sorted members / means / order key
  int32_t* big_list;     // bins of 17 .. kWarpBin votes: one warp each (hough_finish_big_kernel)
  int32_t* huge_list;    // larger bins: one CTA each (hough_finish_huge_kernel)
  int32_t* list_count;   // [0] big, [1] huge
  int64_t big_cap;
};

constexpr int kSmallBin = 16;    // bins up to this size are finished by a single thread
constexpr int kWarpBin = 1024;   // ... up to this size by one warp, above by one CTA
constexpr int kFinishThreads = 128;

__device__ __forceinline__ int64_t order_key(const FinishArgs& a, int64_t rec, int first) {
  const uint32_t base = a.base_bin[first];
  int code = a.bin_code[rec];
  const Bins4 b = a.bins;
  const int cs = code % b.s; code /= b.s;
  const int ct = code % b.t; code /= b.t;
  const int cy = code % b.y; code /= b.y;
  const int cx = code;
  const int o = ((cx - static_cast<int>(base & 0xFF)) << 3) | ((cy - static_cast<int>((base >> 8) & 0xFF)) << 2) |
                ((ct - static_cast<int>((base >> 16) & 0xFF)) << 1) | (cs - static_cast<int>(base >> 24));
  return static_cast<int64_t>(first) * 16 + o;
}

// The six quantities PoseBin averages for one member: x, y, angle, scale (estimate_object_pose) and the
// model image's (w, h) - two contiguous rows, no dependent gathers.
struct Member6 {
  double v[6];
};
__device__ __forceinline__ Member6 load_member(const FinishArgs& a, int m) {
  const double2* p = reinterpret_cast<const double2*>(a.pose) + static_cast<int64_t>(m) * 2;
  const double2 p0 = __ldg(p), p1 = __ldg(p + 1), sz = __ldg(reinterpret_cast<const double2*>(a.match_size) + m);
  return Member6{{p0.x, p0.y, p1.x, p1.y, sz.x, sz.y}};
}
// PoseBin.update_* (PoseBin.py:19-43): mean <- (mean * votes + new) / (votes + 1), votes = j members so far.
// The six means of a bin divide by the same small integer, so the division is a correctly rounded
// reciprocal (rcp = __drcp_rn(j + 1), once per member) followed by Markstein's sequence
//   q = rn(a * rcp);  r = a - (j + 1) * q (exact in one FMA);  result = rn(q + r * rcp)
// which returns the correctly rounded quotient rn(a / (j + 1)) for finite normal operands - the value IEEE
// division gives (checked against exact rational arithmetic on 3e5 random operands, DESIGN.md §4) - at a
// quarter of the instructions of six full divisions.
__device__ __forceinline__ double running_mean(double mean, double v, int j, double rcp) {
  const double a = __dadd_rn(__dmul_rn(mean, static_cast<double>(j)), v);
  const double q = __dmul_rn(a, rcp);
  const double r = __fma_rn(-static_cast<double>(j + 1), q, a);
  return __fma_rn(r, rcp, q);
}

// One THREAD per bin (almost all bins hold a handful of votes): sort the members by match id (the
// reference's append order) in a private strip of shared memory, run the six sequential running means
// of PoseBin.update_posebin and compute the insertion-order key.  Single-vote bins (the majority) skip
// the sort; larger bins are queued for the warp-per-bin and CTA-per-bin kernels.
__global__ void __launch_bounds__(kFinishThreads, 10) hough_finish_kernel(const FinishArgs a) {
  __shared__ int s_m[kSmallBin][kFinishThreads + 1];  // column = thread: conflict-free for equal rows
  int64_t n_bins = a.counters[0];
  if (n_bins > a.cap_bins || a.counters[3]) n_bins = 0;
  const int t = threadIdx.x;
  for (int64_t rec = static_cast<int64_t>(blockIdx.x) * blockDim.x + t; rec < n_bins;
       rec += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int cnt = a.bin_count[rec];
    if (cnt < a.detail_min_count) continue;
    if (cnt > kSmallBin) {
      const bool huge = cnt > kWarpBin;
      const int slot = atomicAdd(a.list_count + (huge ? 1 : 0), 1);
      if (slot < a.big_cap) (huge ? a.huge_list : a.big_list)[slot] = static_cast<int32_t>(rec);
      continue;
    }
    const int off = a.bin_offset[rec];
    SOD_DCHECK(off >= 0 && cnt >= 1);
    double mean[6];
    int first;
    if (cnt == 1) {
      first = a.members_raw[off];
      a.members[off] = first;
      const Member6 v = load_member(a, first);
#pragma unroll
      for (int c = 0; c < 6; ++c) mean[c] = v.v[c];
    } else {
      for (int i = 0; i < cnt; ++i) {  // insertion sort: a few elements, runtime bounds, no wasted slots
        const int x = a.members_raw[off + i];
        int j = i;
        while (j > 0 && s_m[j - 1][t] > x) {
          s_m[j][t] = s_m[j - 1][t];
          --j;
        }
        s_m[j][t] = x;
      }
      first = s_m[0][t];
      for (int j = 0; j < cnt; ++j) {
        const int m = s_m[j][t];
        a.members[off + j] = m;
        const Member6 v = load_member(a, m);
        const double rcp = __drcp_rn(static_cast<double>(j + 1));
#pragma unroll
        for (int c = 0; c < 6; ++c) mean[c] = j == 0 ? v.v[c] : running_mean(mean[c], v.v[c], j, rcp);
      }
    }
#pragma unroll
    for (int c = 0; c < 6; ++c) a.bin_mean[rec * 6 + c] = mean[c];
    a.bin_order[rec] = order_key(a, rec, first);
  }
}

// One component of one member: x, y, angle, scale from the pose row, w, h from the model image size.
__device__ __forceinline__ double member_component(const FinishArgs& a, int m, int c) {
  return c < 4 ? __ldg(a.pose + static_cast<int64_t>(m) * 4 + c) : __ldg(a.match_size + static_cast<int64_t>(m) * 2 + (c - 4));
}

// The sequential means of sorted member lists by one warp: lane = (list k = lane / 6, component c = lane % 6),
// five lists side by side (lanes 30, 31 idle).  Every lane runs ONE recurrence; the value of the next member is
// fetched while the current step's dependent multiply / add / divide chain runs.
__device__ __forceinline__ void warp_means5(const FinishArgs& a, const int32_t* const (&sorted)[5], const int (&cnt)[5],
                                            const int64_t (&rec)[5], int lane) {
  const int k = lane / 6, c = lane - k * 6;
  const int32_t* mine = nullptr;
  int n = 0;
  int64_t my_rec = 0;
#pragma unroll
  for (int i = 0; i < 5; ++i)
    if (k == i) { mine = sorted[i]; n = cnt[i]; my_rec = rec[i]; }
  if (k >= 5) n = 0;
  // The values of the next eight members are requested while the current eight are folded in: a step of the
  // chain is ~100 cycles of dependent arithmetic, a random row read from L2 / HBM several hundred.
  constexpr int kAhead = 8;
  double mean = 0.0;
  double cur[kAhead];
#pragma unroll
  for (int k = 0; k < kAhead; ++k) cur[k] = k < n ? member_component(a, mine[k], c) : 0.0;
  for (int base = 0; base < n; base += kAhead) {
    double nxt[kAhead];
#pragma unroll
    for (int k = 0; k < kAhead; ++k) nxt[k] = base + kAhead + k < n ? member_component(a, mine[base + kAhead + k], c) : 0.0;
#pragma unroll
    for (int k = 0; k < kAhead; ++k) {
      const int j = base + k;
      if (j < n) mean = j == 0 ? cur[k] : running_mean(mean, cur[k], j, __drcp_rn(static_cast<double>(j + 1)));
    }
#pragma unroll
    for (int k = 0; k < kAhead; ++k) cur[k] = nxt[k];
  }
  if (n > 0) {
    a.bin_mean[my_rec * 6 + c] = mean;
    if (c == 0) a.bin_order[my_rec] = order_key(a, my_rec, mine[0]);
  }
}

// Bins of 17 .. kWarpBin votes: a warp takes five of them; each is sorted by the whole warp in a
// shared-memory copy (bitonic), then the five mean chains run side by side.
constexpr int kBigWarps = 4;
__global__ void __launch_bounds__(kBigWarps * 32) hough_finish_big_kernel(const FinishArgs a) {
  __shared__ int32_t s_raw[kBigWarps][kWarpBin];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t warp = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  int64_t n_big = a.list_count[0];
  if (n_big > a.big_cap) n_big = a.big_cap;
  for (int64_t b0 = warp * 5; b0 < n_big; b0 += n_warps * 5) {
    const int32_t* sorted[5];
    int cnt[5];
    int64_t rec[5];
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      sorted[i] = nullptr; cnt[i] = 0; rec[i] = 0;
      if (b0 + i >= n_big) continue;
      rec[i] = a.big_list[b0 + i];
      const int off = a.bin_offset[rec[i]];
      cnt[i] = a.bin_count[rec[i]];
      const int32_t* raw = a.members_raw + off;
      int32_t* out = a.members + off;
      SOD_DCHECK(cnt[i] <= kWarpBin);
      // bitonic sort of the bin's ids in the warp's strip of shared memory, padded with INT_MAX to a power of
      // two: n log^2 n / 64 compare-exchanges per lane instead of the n^2 / 32 compares of a rank sort
      int padded = 32;
      while (padded < cnt[i]) padded <<= 1;
      int32_t* sm = s_raw[w];
      for (int j = lane; j < padded; j += 32) sm[j] = j < cnt[i] ? raw[j] : INT_MAX;
      __syncwarp();
      for (int k = 2; k <= padded; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
          for (int t = lane; t < (padded >> 1); t += 32) {
            const int lo = ((t & ~(j - 1)) << 1) | (t & (j - 1)), hi = lo | j;
            const int32_t x = sm[lo], y = sm[hi];
            if ((x > y) == ((lo & k) == 0)) {
              sm[lo] = y;
              sm[hi] = x;
            }
          }
          __syncwarp();
        }
      }
      for (int j = lane; j < cnt[i]; j += 32) out[j] = sm[j];
      __syncwarp();
      sorted[i] = out;
    }
    warp_means5(a, sorted, cnt, rec, lane);
  }
}

// One CTA per bin of more than kWarpBin votes (a dominant object in a single Hough space can put 10^4-10^5
// matches into one bin).  Match ids are distinct, so the sort is a bitmap: windows of kWindowBits
// consecutive ids are marked in shared memory and read back in order - O(votes + id range) instead of the
// O(votes^2) of a rank sort.  The running means stay one sequential chain (the reference's recurrence is
// order dependent), fed by warp 0 through warp_means.
constexpr int kHugeThreads = 1024;
constexpr int kWindowWords = 32768;                 // 128 KB of shared memory
constexpr int64_t kWindowBits = int64_t(kWindowWords) * 32;

__global__ void __launch_bounds__(kHugeThreads, 1) hough_finish_huge_kernel(const FinishArgs a) {
  extern __shared__ uint32_t bitmap[];
  __shared__ int s_lo, s_hi, s_warp_tot[32], s_base;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int64_t n_huge = a.list_count[1];
  if (n_huge > a.big_cap) n_huge = a.big_cap;
  for (int64_t b = blockIdx.x; b < n_huge; b += gridDim.x) {
    const int64_t rec = a.huge_list[b];
    const int off = a.bin_offset[rec], cnt = a.bin_count[rec];
    const int32_t* raw = a.members_raw + off;
    int32_t* out = a.members + off;
    if (tid == 0) { s_lo = INT_MAX; s_hi = INT_MIN; s_base = 0; }
    __syncthreads();
    int lo = INT_MAX, hi = INT_MIN;
    for (int i = tid; i < cnt; i += kHugeThreads) {
      const int x = raw[i];
      lo = min(lo, x);
      hi = max(hi, x);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
      hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    if (lane == 0) { atomicMin(&s_lo, lo); atomicMax(&s_hi, hi); }
    __syncthreads();
    const int id_lo = s_lo, id_hi = s_hi;
    for (int64_t w0 = id_lo; w0 <= id_hi; w0 += kWindowBits) {
      for (int i = tid; i < kWindowWords; i += kHugeThreads) bitmap[i] = 0u;
      __syncthreads();
      for (int i = tid; i < cnt; i += kHugeThreads) {
        const int64_t d = static_cast<int64_t>(raw[i]) - w0;
        if (d >= 0 && d < kWindowBits) atomicOr(&bitmap[d >> 5], 1u << (d & 31));
      }
      __syncthreads();
      // every thread owns kWindowWords / kHugeThreads consecutive words: count, scan over the CTA, emit
      constexpr int kPer = kWindowWords / kHugeThreads;
      int mine = 0;
#pragma unroll 4
      for (int k = 0; k < kPer; ++k) mine += __popc(bitmap[tid * kPer + k]);
      int pos = s_base + cta_exclusive_scan(mine, s_warp_tot);
      for (int k = 0; k < kPer; ++k) {
        uint32_t word = bitmap[tid * kPer + k];
        while (word) {
          const int bit = __ffs(word) - 1;
          word &= word - 1;
          SOD_DCHECK(pos < cnt);
          out[pos++] = static_cast<int32_t>(w0 + (static_cast<int64_t>(tid * kPer + k) << 5) + bit);
        }
      }
      __syncthreads();
      if (tid == kHugeThreads - 1) s_base = pos;  // the last thread's end = the window's total
      __syncthreads();
    }
    __threadfence_block();
    __syncthreads();
    if (warp == 0) {
      const int32_t* const sorted[5] = {out, nullptr, nullptr, nullptr, nullptr};
      const int cnts[5] = {cnt, 0, 0, 0, 0};
      const int64_t recs[5] = {rec, 0, 0, 0, 0};
      warp_means5(a, sorted, cnts, recs, lane);
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------ compaction
constexpr int kCompactThreads = 1024;

__global__ void __launch_bounds__(kCompactThreads)
compact_count_kernel(const int32_t* __restrict__ idx, const uint8_t* __restrict__ pass, int64_t n,
                     int32_t t_lo, int32_t t_hi, int32_t* __restrict__ block_counts) {
  __shared__ int s;
  if (threadIdx.x == 0) s = 0;
  __syncthreads();
  const int64_t i = static_cast<int64_t>(blockIdx.x) * kCompactThreads + threadIdx.x;
  bool keep = i < n && pass[i];
  if (keep) {
    const int32_t t = idx[i * 2];
    keep = t >= t_lo && t < t_hi;
  }
  const unsigned b = __ballot_sync(0xffffffffu, keep);
  if ((threadIdx.x & 31) == 0 && b) atomicAdd(&s, __popc(b));
  __syncthreads();
  if (threadIdx.x == 0) block_counts[blockIdx.x] = s;
}

__global__ void __launch_bounds__(kCompactThreads)
compact_write_kernel(const int32_t* __restrict__ idx, const uint8_t* __restrict__ pass, int64_t n,
                     int32_t t_lo, int32_t t_hi, const int32_t* __restrict__ block_off,
                     int32_t* __restrict__ match_q, int32_t* __restrict__ match_t) {
  __shared__ int warp_base[kCompactThreads / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t i = static_cast<int64_t>(blockIdx.x) * kCompactThreads + threadIdx.x;
  bool keep = i < n && pass[i];
  int32_t t = 0;
  if (keep) {
    t = idx[i * 2];
    keep = t >= t_lo && t < t_hi;
  }
  const unsigned b = __ballot_sync(0xffffffffu, keep);
  if (lane == 0) warp_base[warp] = __popc(b);
  __syncthreads();
  if (warp == 0) {
    const int v = warp_base[lane];
    warp_base[lane] = warp_inclusive_scan(v) - v;
  }
  __syncthreads();
  if (keep) {
    const int pos = block_off[blockIdx.x] + warp_base[warp] + __popc(b & ((1u << lane) - 1u));
    SOD_DCHECK(pos >= 0 && pos < n);
    match_q[pos] = static_cast<int32_t>(i);
    match_t[pos] = t;
  }
}

size_t align256(size_t x) { return (x + 255) & ~static_cast<size_t>(255); }

struct HoughWs {
  int32_t *group_of, *group_count, *group_off, *group_rank, *grouped, *members_raw, *ticket, *big_list, *huge_list;
  int32_t* scan_tiles;
  uint32_t *grouped_base, *rank;
  uint16_t* creator;
  double* match_size;
  int64_t big_cap;
  size_t bytes;
};

// Sub-counters per Hough space of the counting sort (hough_pose_kernel): up to 16, as long as all of them
// fit 65,536 counters - scenes with many spaces spread their atomics by themselves.
int group_sub_shift(int64_t groups) {
  int shift = 0;
  while (shift < 4 && (groups << (shift + 1)) <= 65536) ++shift;
  return shift;
}

HoughWs carve_hough_ws(void* base, int64_t m, int64_t groups, int64_t cap_votes) {
  HoughWs w;
  groups <<= group_sub_shift(groups);  // group_count / group_off / the scan hold one entry per sub-counter
  size_t o = 0;
  auto take = [&](size_t bytes) {
    void* p = base ? static_cast<char*>(base) + o : nullptr;
    o += align256(bytes);
    return p;
  };
  w.ticket = static_cast<int32_t*>(take(256));
  w.group_of = static_cast<int32_t*>(take(m * 4));
  w.group_count = static_cast<int32_t*>(take((groups + 1) * 4));
  w.group_off = static_cast<int32_t*>(take((groups + 1) * 4));
  w.group_rank = static_cast<int32_t*>(take(m * 4));
  w.scan_tiles = static_cast<int32_t*>(take(2 * ((groups + kScanTile - 1) / kScanTile + 2) * 4));
  w.grouped = static_cast<int32_t*>(take(m * 4));
  w.grouped_base = static_cast<uint32_t*>(take(m * 4));
  w.rank = static_cast<uint32_t*>(take(m * 16 * 4));
  w.creator = static_cast<uint16_t*>(take(m * 2));
  w.match_size = static_cast<double*>(take(m * 2 * 8));
  w.members_raw = static_cast<int32_t*>(take(cap_votes * 4));
  w.big_cap = cap_votes / (kSmallBin + 1) + 1;
  w.big_list = static_cast<int32_t*>(take(w.big_cap * 4));
  w.huge_list = static_cast<int32_t*>(take((cap_votes / (kWarpBin + 1) + 1) * 4));
  w.bytes = o;
  return w;
}

}  // namespace
}  // namespace sod

using namespace sod;

extern "C" {

size_t sod_compact_scratch_bytes(int64_t n_query) {
  const int64_t blocks = n_query <= 0 ? 1 : (n_query + kCompactThreads - 1) / kCompactThreads;
  return static_cast<size_t>(2 * (blocks + 1)) * 4;
}

int sod_compact_matches(const int32_t* idx, const uint8_t* pass, int64_t n_query, int32_t t_lo,
                        int32_t t_hi, int32_t* match_q, int32_t* match_t, int32_t* n_out,
                        void* scratch, sod_stream_t stream) {
  SOD_CHECK_ARG(n_query >= 0, "n_query < 0");
  SOD_CHECK_ARG(n_out, "null n_out");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (n_query == 0) {
    SOD_CHECK_CUDA(cudaMemsetAsync(n_out, 0, 4, st));
    return SOD_OK;
  }
  SOD_CHECK_ARG(idx && pass && match_q && match_t && scratch, "null pointer");
  const int64_t blocks = (n_query + kCompactThreads - 1) / kCompactThreads;
  int32_t* counts = static_cast<int32_t*>(scratch);
  int32_t* offs = counts + blocks + 1;
  compact_count_kernel<<<static_cast<unsigned>(blocks), kCompactThreads, 0, st>>>(idx, pass, n_query, t_lo,
                                                                                  t_hi, counts);
  SOD_CHECK_LAUNCH("compact_count_kernel");
  exclusive_scan_kernel<<<1, 1024, 0, st>>>(counts, blocks, offs, n_out, nullptr);
  SOD_CHECK_LAUNCH("exclusive_scan_kernel");
  compact_write_kernel<<<static_cast<unsigned>(blocks), kCompactThreads, 0, st>>>(
      idx, pass, n_query, t_lo, t_hi, offs, match_q, match_t);
  SOD_CHECK_LAUNCH("compact_write_kernel");
  return SOD_OK;
}

int sod_estimate_pose(const sod_scene* scene, const int32_t* match_q, const int32_t* match_t,
                      int64_t n_matches, int32_t bins, const int32_t* sigma_lut, double* pose,
                      uint32_t* base_bin, uint8_t* near_edge, sod_stream_t stream) {
  SOD_CHECK_ARG(scene && n_matches >= 0, "bad arguments");
  if (n_matches == 0) return SOD_OK;
  SOD_CHECK_ARG(bins >= 1 && bins <= 255, "bins out of range");
  SOD_CHECK_ARG(match_q && match_t && sigma_lut && pose && base_bin, "null pointer");
  SOD_CHECK_ARG(scene->query.xy && scene->query.angle && scene->query.octave && scene->model.xy &&
                    scene->model.angle && scene->model.octave && scene->model_image &&
                    scene->image_centroid && scene->frame_wh && scene->groups_per_frame >= 1,
                "null scene array");
  PoseArgs pa;
  pa.sc = *scene;
  pa.match_q = match_q; pa.match_t = match_t; pa.n_dev = nullptr; pa.n_cap = n_matches;
  pa.bins = Bins4{bins, bins, bins, bins}; pa.sigma_lut = sigma_lut; pa.pose = pose; pa.base_bin = base_bin;
  pa.near_edge = near_edge; pa.counters = nullptr; pa.group_of = nullptr; pa.group_count = nullptr;
  pa.group_rank = nullptr; pa.match_size = nullptr; pa.group_shift = 0;
  const int threads = 256;
  hough_pose_kernel<<<static_cast<unsigned>((n_matches + threads - 1) / threads), threads, 0,
                      static_cast<cudaStream_t>(stream)>>>(pa);
  SOD_CHECK_LAUNCH("hough_pose_kernel");
  return SOD_OK;
}

int sod_pose_bin_index(const double* pose, int64_t n, int32_t bins, int32_t width, int32_t height,
                       const int32_t* sigma_lut, uint32_t* base_bin, sod_stream_t stream) {
  SOD_CHECK_ARG(n >= 0 && bins >= 1 && bins <= 255 && width > 0 && height > 0, "bad arguments");
  if (n == 0) return SOD_OK;
  SOD_CHECK_ARG(pose && sigma_lut && base_bin, "null pointer");
  const int threads = 256;
  pose_bin_index_kernel<<<static_cast<unsigned>((n + threads - 1) / threads), threads, 0,
                          static_cast<cudaStream_t>(stream)>>>(pose, n, bins, width, height, sigma_lut,
                                                               base_bin);
  SOD_CHECK_LAUNCH("pose_bin_index_kernel");
  return SOD_OK;
}

size_t sod_hough_workspace_bytes(int64_t n_matches, int64_t n_groups) {
  if (n_matches < 0) n_matches = 0;
  if (n_groups < 1) n_groups = 1;
  return carve_hough_ws(nullptr, n_matches, n_groups, n_matches * 16).bytes + 256;
}

int sod_hough_vote(const sod_scene* scene, const int32_t* match_q, const int32_t* match_t,
                   int64_t n_matches, const int32_t* n_matches_dev, int32_t bins,
                   const int32_t* sigma_lut, int32_t detail_min_count, const sod_hough_out* out,
                   void* workspace, size_t workspace_bytes, sod_stream_t stream) {
  return sod_hough_vote_dims(scene, match_q, match_t, n_matches, n_matches_dev, bins, bins, bins, bins, sigma_lut,
                             detail_min_count, out, workspace, workspace_bytes, stream);
}

int sod_hough_vote_dims(const sod_scene* scene, const int32_t* match_q, const int32_t* match_t,
                        int64_t n_matches, const int32_t* n_matches_dev, int32_t bins_x, int32_t bins_y,
                        int32_t bins_theta, int32_t bins_sigma, const int32_t* sigma_lut,
                        int32_t detail_min_count, const sod_hough_out* out, void* workspace,
                        size_t workspace_bytes, sod_stream_t stream) {
  SOD_CHECK_ARG(scene && out, "null scene/out");
  SOD_CHECK_ARG(n_matches >= 0 && n_matches < (int64_t(1) << 27), "n_matches out of range");
  SOD_CHECK_ARG(bins_x >= 1 && bins_y >= 1 && bins_theta >= 1 && bins_sigma >= 1, "bins < 1");
  const Bins4 bins{bins_x, bins_y, bins_theta, bins_sigma};
  constexpr int64_t kMaxCounters = int64_t(SOD_MAX_BINS) * SOD_MAX_BINS * SOD_MAX_BINS * SOD_MAX_BINS;
  if (bins_x > 255 || bins_y > 255 || bins_theta > 255 || bins_sigma > 255 ||
      int64_t(bins_x) * bins_y * bins_theta * bins_sigma > kMaxCounters) {
    set_error("bins = %d x %d x %d x %d: the shared-memory histogram holds at most %d^4 counters", bins_x, bins_y,
              bins_theta, bins_sigma, SOD_MAX_BINS);
    return SOD_ERR_UNSUPPORTED;
  }
  SOD_CHECK_ARG(out->counters, "null counters");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  SOD_CHECK_CUDA(cudaMemsetAsync(out->counters, 0, 8 * sizeof(int32_t), st));
  if (n_matches == 0) return SOD_OK;
  const int64_t n_groups = static_cast<int64_t>(scene->n_frames) * scene->groups_per_frame;
  SOD_CHECK_ARG(scene->n_frames >= 1 && scene->groups_per_frame >= 1 && n_groups < (int64_t(1) << 30),
                "bad frame/group counts");
  SOD_CHECK_ARG(match_q && match_t && sigma_lut && workspace, "null pointer");
  SOD_CHECK_ARG(scene->query.xy && scene->query.angle && scene->query.octave && scene->model.xy &&
                    scene->model.angle && scene->model.octave && scene->model_image &&
                    scene->image_centroid && scene->image_size && scene->frame_wh,
                "null scene array");
  SOD_CHECK_ARG(out->pose && out->base_bin && out->near_edge && out->bin_group && out->bin_code &&
                    out->bin_count && out->bin_offset && out->bin_order && out->bin_mean && out->members,
                "null output array");
  SOD_CHECK_ARG(out->cap_votes < (int64_t(1) << 31) && out->cap_bins < (int64_t(1) << 31), "capacity >= 2^31");
  SOD_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "workspace must be 256-byte aligned");
  const int64_t raw_cap = out->cap_votes < n_matches * 16 ? out->cap_votes : n_matches * 16;
  const HoughWs w = carve_hough_ws(workspace, n_matches, n_groups, raw_cap);
  SOD_CHECK_ARG(workspace_bytes >= w.bytes, "workspace too small: %zu < %zu", workspace_bytes, w.bytes);
  const int sms = device_sm_count();
  if (sms <= 0) return SOD_ERR_CUDA;

  const int group_shift = group_sub_shift(n_groups);
  const int64_t n_sub = n_groups << group_shift;
  SOD_CHECK_CUDA(cudaMemsetAsync(w.group_count, 0, (n_sub + 1) * 4, st));
  SOD_CHECK_CUDA(cudaMemsetAsync(w.ticket, 0, 12, st));  // [0] vote ticket, [1] big-bin count, [2] huge-bin count
  PoseArgs pa;
  pa.sc = *scene;
  pa.match_q = match_q; pa.match_t = match_t; pa.n_dev = n_matches_dev; pa.n_cap = n_matches;
  pa.bins = bins; pa.sigma_lut = sigma_lut; pa.pose = out->pose; pa.base_bin = out->base_bin;
  pa.near_edge = out->near_edge; pa.counters = out->counters; pa.group_of = w.group_of;
  pa.group_count = w.group_count; pa.group_rank = w.group_rank; pa.match_size = w.match_size;
  pa.group_shift = group_shift;
  const int threads = 256;
  int64_t blocks = (n_matches + threads - 1) / threads;
  if (blocks > static_cast<int64_t>(sms) * 16) blocks = static_cast<int64_t>(sms) * 16;
  stage_begin(SOD_STAGE_HOUGH_PREP, st);
  hough_pose_kernel<<<static_cast<unsigned>(blocks), threads, 0, st>>>(pa);
  SOD_CHECK_LAUNCH("hough_pose_kernel");
  SOD_CHECK_CUDA(device_exclusive_scan(w.group_count, n_sub, w.group_off, w.scan_tiles, st));
  group_scatter_kernel<<<static_cast<unsigned>(blocks), threads, 0, st>>>(
      w.group_of, w.group_rank, out->base_bin, n_matches_dev, n_matches, w.group_off, w.grouped, w.grouped_base);
  SOD_CHECK_LAUNCH("group_scatter_kernel");
  stage_end(SOD_STAGE_HOUGH_PREP, st);

  VoteArgs va;
  va.group_off = w.group_off; va.grouped = w.grouped; va.base_bin = w.grouped_base; va.rank = w.rank; va.creator = w.creator;
  va.n_groups = n_groups; va.group_shift = group_shift; va.bins = bins; va.ticket = w.ticket; va.counters = out->counters; va.bin_group = out->bin_group;
  va.bin_code = out->bin_code; va.bin_count = out->bin_count; va.bin_offset = out->bin_offset;
  va.members_raw = w.members_raw; va.cap_bins = out->cap_bins; va.cap_votes = raw_cap;
  const size_t hist_bytes = static_cast<size_t>(bins.total()) * sizeof(uint32_t);
  SOD_CHECK_CUDA(cudaFuncSetAttribute(hough_vote_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      static_cast<int>(hist_bytes)));  // per device, hence at every launch
  int64_t group_chunk = n_groups / (static_cast<int64_t>(sms) * 8);
  group_chunk = group_chunk < 1 ? 1 : (group_chunk > kGroupChunk ? kGroupChunk : group_chunk);
  va.group_chunk = static_cast<int>(group_chunk);
  const int64_t n_chunks = (n_groups + group_chunk - 1) / group_chunk;
  const int64_t vgrid = n_chunks < sms ? n_chunks : sms;
  {
    StageScope timed(SOD_STAGE_HOUGH_VOTE, st);
    hough_vote_kernel<<<static_cast<unsigned>(vgrid), kVoteThreads, hist_bytes, st>>>(va);
  }
  SOD_CHECK_LAUNCH("hough_vote_kernel");

  FinishArgs fa;
  fa.pose = out->pose; fa.match_size = w.match_size; fa.base_bin = out->base_bin; fa.counters = out->counters;
  fa.bin_code = out->bin_code; fa.bin_count = out->bin_count; fa.bin_offset = out->bin_offset;
  fa.members_raw = w.members_raw; fa.members = out->members; fa.bin_order = out->bin_order;
  fa.bin_mean = out->bin_mean; fa.cap_bins = out->cap_bins; fa.bins = bins;
  fa.detail_min_count = detail_min_count; fa.big_list = w.big_list; fa.huge_list = w.huge_list;
  fa.list_count = w.ticket + 1;
  fa.big_cap = w.big_cap;
  stage_begin(SOD_STAGE_HOUGH_FINISH, st);
  hough_finish_kernel<<<sms * 20, kFinishThreads, 0, st>>>(fa);
  SOD_CHECK_LAUNCH("hough_finish_kernel");
  hough_finish_big_kernel<<<sms * 8, kBigWarps * 32, 0, st>>>(fa);
  SOD_CHECK_LAUNCH("hough_finish_big_kernel");
  constexpr int kHugeSmem = kWindowWords * 4;
  SOD_CHECK_CUDA(cudaFuncSetAttribute(hough_finish_huge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kHugeSmem));
  hough_finish_huge_kernel<<<sms, kHugeThreads, kHugeSmem, st>>>(fa);
  SOD_CHECK_LAUNCH("hough_finish_huge_kernel");
  stage_end(SOD_STAGE_HOUGH_FINISH, st);
  return SOD_OK;
}

}  // extern "C"
