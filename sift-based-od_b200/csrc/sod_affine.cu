// K5: valid-bin selection and per-bin affine verification.
//
// Replaces Main.get_valid_bins / Main.apply_affine_parameters (main.py:121-157), AffineParameters
// (AffineParameters.py:89-113: Gen_A, Gen_b, Calc_x) and remove_outliers (AffineParameters.py:116-160).
//
// The reference's global "while anything changed" loop over all bins is, bin by bin, an independent
// fixed-point iteration (fit and residual test only read the bin's own pairs; SURVEY.md §3.4, T13),
// so one warp owns one bin for all its passes.  The 6x6 normal matrix A^T A of the reference
// (parameter order m1 m2 m3 m4 tx ty) is two interleaved copies of the 3x3 matrix
//   S = sum [x y 1]^T [x y 1]
// so pinv(A^T A) A^T b = ( pinv(S) sum [x y 1]^T u , pinv(S) sum [x y 1]^T v ).  pinv(S) comes from a
// Jacobi eigen-decomposition in fp64 with numpy's default cut-off (rcond = 1e-15 x largest
// eigenvalue), which reproduces the minimum-norm answer on rank-deficient bins (SURVEY Q11).
#include "sod_common.cuh"

namespace sod {
namespace {

struct AffineArgs {
  sod_scene sc;
  const int32_t* match_q;
  const int32_t* match_t;
  const int32_t* hough_counters;
  const int32_t* bin_group;
  const int32_t* bin_code;
  const int32_t* bin_count;
  const int32_t* bin_offset;
  const int32_t* members;
  int64_t cap_bins;
  int bins, vote_threshold, affine_threshold, max_passes;
  double factor_x, factor_y;
  sod_affine_out out;
};

__global__ void affine_select_kernel(const AffineArgs a) {
  int64_t n_bins = a.hough_counters[0];
  if (n_bins > a.cap_bins || a.hough_counters[3]) n_bins = 0;
  // one atomic per warp: the surviving bins of 32 consecutive records take consecutive slots (a stress scene
  // selects 1.6 M bins: as single same-address atomics with return they were 0.17 ms)
  const unsigned lane = threadIdx.x & 31u;
  for (int64_t base = static_cast<int64_t>(blockIdx.x) * blockDim.x + (threadIdx.x & ~31u); base < n_bins;
       base += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t rec = base + lane;
    const bool take = rec < n_bins && a.bin_count[rec] >= a.vote_threshold;
    const unsigned takers = __ballot_sync(0xffffffffu, take);
    if (!takers) continue;
    const int leader = __ffs(takers) - 1;
    int first = 0;
    if (static_cast<int>(lane) == leader) first = atomicAdd(&a.out.counters[0], __popc(takers));
    first = __shfl_sync(0xffffffffu, first, leader);
    if (take) {
      const int v = first + __popc(takers & ((1u << lane) - 1u));
      if (v < a.out.cap_valid)
        a.out.valid_bin[v] = static_cast<int32_t>(rec);
      else
        a.out.counters[1] = 1;
    }
  }
}

// Cyclic Jacobi on a symmetric 3x3: A -> diag(w), columns of V are the eigenvectors.
__device__ void jacobi3(double (&A)[3][3], double (&V)[3][3]) {
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) V[i][j] = i == j ? 1.0 : 0.0;
  for (int sweep = 0; sweep < 16; ++sweep) {
    const double off = fabs(A[0][1]) + fabs(A[0][2]) + fabs(A[1][2]);
    const double diag = fabs(A[0][0]) + fabs(A[1][1]) + fabs(A[2][2]);
    if (off <= 1e-300 || off <= 1e-22 * diag) break;
#pragma unroll
    for (int pq = 0; pq < 3; ++pq) {
      const int p = pq == 2 ? 1 : 0, q = pq == 0 ? 1 : 2;
      const double apq = A[p][q];
      if (apq == 0.0) continue;
      const double theta = (A[q][q] - A[p][p]) / (2.0 * apq);
      const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
      const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
      const int r = 3 - p - q;  // the untouched index
      const double app = A[p][p], aqq = A[q][q], arp = A[r][p], arq = A[r][q];
      A[p][p] = app - t * apq;
      A[q][q] = aqq + t * apq;
      A[p][q] = A[q][p] = 0.0;
      A[r][p] = A[p][r] = c * arp - s * arq;
      A[r][q] = A[q][r] = s * arp + c * arq;
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        const double vip = V[i][p], viq = V[i][q];
        V[i][p] = c * vip - s * viq;
        V[i][q] = s * vip + c * viq;
      }
    }
  }
}

// pinv(S) applied to the two right-hand sides: S = [[sxx,sxy,sx],[sxy,syy,sy],[sx,sy,n]].
// Returns 1 if S is numerically singular (smallest |eigenvalue| <= 1e-10 x largest).
__device__ __forceinline__ int solve_affine(double sxx, double sxy, double sx, double syy, double sy,
                                            double sn, const double (&ru)[3], const double (&rv)[3],
                                            double (&pu)[3], double (&pv)[3]) {
  double A[3][3] = {{sxx, sxy, sx}, {sxy, syy, sy}, {sx, sy, sn}};
  double V[3][3];
  jacobi3(A, V);
  const double wv[3] = {A[0][0], A[1][1], A[2][2]};
  const double wmax = fmax(fabs(wv[0]), fmax(fabs(wv[1]), fabs(wv[2])));
  const double wmin = fmin(fabs(wv[0]), fmin(fabs(wv[1]), fabs(wv[2])));
  const double cut = 1e-15 * wmax;  // numpy.linalg.pinv default rcond
#pragma unroll
  for (int i = 0; i < 3; ++i) pu[i] = pv[i] = 0.0;
#pragma unroll
  for (int e = 0; e < 3; ++e) {
    if (!(fabs(wv[e]) > cut)) continue;
    const double du = (V[0][e] * ru[0] + V[1][e] * ru[1] + V[2][e] * ru[2]) / wv[e];
    const double dv = (V[0][e] * rv[0] + V[1][e] * rv[1] + V[2][e] * rv[2]) / wv[e];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      pu[i] += V[i][e] * du;
      pv[i] += V[i][e] * dv;
    }
  }
  return wmin <= 1e-10 * wmax ? 1 : 0;
}

constexpr int kSmallAffine = 32;  // bins up to this size are verified by a single thread

// remove_outliers keeps a pair unless |u_AP - u| > x_ref or |v_AP - v| > y_ref (AffineParameters.py:152).
// The fitted parameters agree with numpy's pinv to ~1e-12 relative on well-conditioned bins (more on
// near-singular ones), so a residual this close to its limit could be decided the other way by the
// reference; such decisions are counted (counters[3], status bit 2), never altered.
__device__ __forceinline__ bool residual_on_edge(double du, double dv, double x_ref, double y_ref) {
  return fabs(du - x_ref) <= 1e-9 * x_ref + 1e-7 || fabs(dv - y_ref) <= 1e-9 * y_ref + 1e-7;
}

// Residual limits (x_ref, y_ref) of a bin: remove_outliers thresholds use pose[3], the sigma BIN INDEX
// (AffineParameters.py:120-121).  A factor <= 0 disables its limit.
__device__ __forceinline__ double2 residual_limits(const AffineArgs& a, int rec) {
  const int frame = a.bin_group[rec] / a.sc.groups_per_frame;
  SOD_DCHECK(frame >= 0 && frame < a.sc.n_frames);
  const int isigma = a.bin_code[rec] % a.bins;
  const double inf = __longlong_as_double(0x7ff0000000000000ll);
  return make_double2(
      a.factor_x > 0 ? __ddiv_rn(static_cast<double>(a.sc.frame_wh[2 * frame] * isigma), a.factor_x) : inf,
      a.factor_y > 0 ? __ddiv_rn(static_cast<double>(a.sc.frame_wh[2 * frame + 1] * isigma), a.factor_y) : inf);
}

// A bin whose members lie past cap_votes (member_keep was sized for another Hough result) is not verified:
// reject_bin flags the overflow and gives the bin no votes.
__device__ __forceinline__ bool members_past_capacity(const AffineArgs& a, int off, int cnt) {
  return static_cast<int64_t>(off) + cnt > a.out.cap_votes;
}
__device__ __forceinline__ void reject_bin(const AffineArgs& a, int64_t v) {
  a.out.counters[1] = 1;
  a.out.votes[v] = 0;
  a.out.status[v] = 0;
}

// (x, y) of the model point and (u, v) of the query point of member j: three dependent gathers
// (member -> match -> keypoint).
__device__ __forceinline__ float4 pair_coords(const AffineArgs& a, const int32_t* mem, int j) {
  const int m = mem[j];
  SOD_DCHECK(m >= 0 && a.match_t[m] >= 0 && a.match_t[m] < a.sc.model.n && a.match_q[m] >= 0 &&
             a.match_q[m] < a.sc.query.n);
  const float2 pm = reinterpret_cast<const float2*>(a.sc.model.xy)[a.match_t[m]];
  const float2 pq = reinterpret_cast<const float2*>(a.sc.query.xy)[a.match_q[m]];
  return make_float4(pm.x, pm.y, pq.x, pq.y);
}

// |u_AP - u| of a pair for the fitted coordinate u_AP = ma * x + mb * y + t, in the reference's operation
// order (AffineParameters.py:128-155): (m1, m2, tx) against the query's u, (m3, m4, ty) against its v.
__device__ __forceinline__ double fit_residual(double ma, double mb, double t, double x, double y, float u) {
  return fabs(__dadd_rn(__dadd_rn(__dmul_rn(ma, x), __dmul_rn(mb, y)), t) - static_cast<double>(u));
}

// One bin's result: parameters in the order m1 m2 m3 m4 tx ty, votes, status word (bit 0 live, 1 singular,
// 2 residual on edge, 8.. passes) and the singular / on-edge counters.
__device__ __forceinline__ void write_bin_result(const AffineArgs& a, int64_t v, const double (&pu)[3],
                                                 const double (&pv)[3], int votes, int live, int singular,
                                                 int on_edge, int passes) {
  double* p = a.out.params + v * 6;
  p[0] = pu[0]; p[1] = pu[1]; p[2] = pv[0]; p[3] = pv[1]; p[4] = pu[2]; p[5] = pv[2];
  a.out.votes[v] = votes;
  a.out.status[v] = live | (singular << 1) | ((on_edge ? 1 : 0) << 2) | (passes << 8);
  if (singular) atomicAdd(&a.out.counters[2], 1);
  if (on_edge) atomicAdd(&a.out.counters[3], on_edge);
}

// One THREAD per small valid bin (the vast majority: random bins with 5-10 votes): the alive set is
// a 32-bit mask, every pass re-gathers the coordinates of the alive pairs.
constexpr int kSmallThreads = 128;
constexpr int kSmallStage = 16;  // pairs of a bin whose coordinates the thread keeps in shared memory

__global__ void __launch_bounds__(kSmallThreads) affine_verify_small_kernel(const AffineArgs a) {
  // coordinates of the bin's first kSmallStage pairs, fetched once (member -> match -> keypoint, three
  // dependent gathers each) instead of twice per pass; [pair][thread] keeps the threads' rows in different banks
  __shared__ float4 s_pairs[kSmallStage][kSmallThreads];
  int64_t n_valid = a.out.counters[0];
  if (n_valid > a.out.cap_valid) n_valid = a.out.cap_valid;
  for (int64_t v = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; v < n_valid;
       v += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int rec = a.out.valid_bin[v];
    SOD_DCHECK(rec >= 0 && rec < a.cap_bins);
    const int cnt = a.bin_count[rec];
    if (cnt > kSmallAffine) continue;
    const int off = a.bin_offset[rec];
    if (members_past_capacity(a, off, cnt)) {
      reject_bin(a, v);
      continue;
    }
    const double2 lim = residual_limits(a, rec);
    const int32_t* mem = a.members + off;
    const int n_stage = cnt < kSmallStage ? cnt : kSmallStage;
#pragma unroll 4
    for (int j = 0; j < n_stage; ++j) s_pairs[j][threadIdx.x] = pair_coords(a, mem, j);
    auto pair_of = [&](int j) -> float4 { return j < kSmallStage ? s_pairs[j][threadIdx.x] : pair_coords(a, mem, j); };
    unsigned alive = cnt >= 32 ? 0xffffffffu : ((1u << cnt) - 1u);
    int n_alive = cnt, passes = 0, live = 0, singular = 0, on_edge = 0;
    double pu[3] = {0, 0, 0}, pv[3] = {0, 0, 0};
    while (true) {
      double sxx = 0, sxy = 0, sx = 0, syy = 0, sy = 0, sn = 0;
      double ru[3] = {0, 0, 0}, rv[3] = {0, 0, 0};
      for (int j = 0; j < cnt; ++j) {
        if (!(alive >> j & 1u)) continue;
        const float4 c = pair_of(j);
        const double x = c.x, y = c.y, u = c.z, w = c.w;
        sxx += x * x; sxy += x * y; sx += x; syy += y * y; sy += y; sn += 1.0;
        ru[0] += x * u; ru[1] += y * u; ru[2] += u; rv[0] += x * w; rv[1] += y * w; rv[2] += w;
      }
      singular |= solve_affine(sxx, sxy, sx, syy, sy, sn, ru, rv, pu, pv);
      int removed = 0;
      for (int j = 0; j < cnt; ++j) {
        if (!(alive >> j & 1u)) continue;
        const float4 c = pair_of(j);
        const double du = fit_residual(pu[0], pu[1], pu[2], c.x, c.y, c.z);
        const double dv = fit_residual(pv[0], pv[1], pv[2], c.x, c.y, c.w);
        on_edge += residual_on_edge(du, dv, lim.x, lim.y) ? 1 : 0;
        if (du > lim.x || dv > lim.y) {
          alive &= ~(1u << j);
          ++removed;
        }
      }
      n_alive -= removed;
      ++passes;
      if (n_alive < a.affine_threshold) break;
      if (removed == 0) { live = 1; break; }
      if (a.max_passes > 0 && passes >= a.max_passes) { live = 1; break; }
    }
    uint8_t* keep = a.out.member_keep + off;
    for (int j = 0; j < cnt; ++j) keep[j] = (alive >> j) & 1u;
    write_bin_result(a, v, pu, pv, n_alive, live, singular, on_edge, passes);
  }
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

constexpr int kAffineWarps = 4;    // warps per CTA of affine_verify_kernel
constexpr int kAffineStage = 512;  // pairs of a bin whose coordinates a warp keeps in shared memory

__global__ void __launch_bounds__(kAffineWarps * 32) affine_verify_kernel(const AffineArgs a) {
  // (x, y) of the model point and (u, v) of the query point of the bin's first kAffineStage pairs: every pass
  // reads each pair twice, and fetching it is three dependent gathers (member -> match -> keypoint) - a
  // 400-pair bin spent its time waiting for them, pass after pass.  Pairs beyond the stage are gathered.
  __shared__ float4 s_xyuv[kAffineWarps][kAffineStage];
  float4* const stage = s_xyuv[threadIdx.x >> 5];
  const int lane = threadIdx.x & 31;
  const int64_t warp = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  int64_t n_valid = a.out.counters[0];
  if (n_valid > a.out.cap_valid) n_valid = a.out.cap_valid;
  // Almost every selected bin is a small one (affine_verify_small_kernel's): the lanes look at a window of up
  // to 32 list entries at a time and the warp then takes the big bins among them in turn.  (One entry per warp and step meant
  // 1.6 M dependent look-ups spread over 3,000 warps at C5: 0.66 ms for 9,000 big bins.)
  // The window shrinks with the list (down to one entry per warp): a warp works through the big bins of its
  // window one after the other, and a short list of mostly big bins (the bench workload: 16,500 entries) must
  // still spread over all warps.
  int width = 32;
  while (width > 1 && n_valid < static_cast<int64_t>(width) * n_warps) width >>= 1;
  for (int64_t v0 = warp * width; v0 < n_valid; v0 += n_warps * width) {
   int rec_l = 0, cnt_l = 0;
   if (lane < width && v0 + lane < n_valid) {
     rec_l = a.out.valid_bin[v0 + lane];
     cnt_l = a.bin_count[rec_l];
   }
   unsigned big = __ballot_sync(0xffffffffu, cnt_l > kSmallAffine);
   while (big) {
    const int src = __ffs(big) - 1;
    big &= big - 1;
    const int64_t v = v0 + src;
    const int rec = __shfl_sync(0xffffffffu, rec_l, src);
    const int cnt = __shfl_sync(0xffffffffu, cnt_l, src);
    const int off = a.bin_offset[rec];
    if (members_past_capacity(a, off, cnt)) {
      if (lane == 0) reject_bin(a, v);
      continue;
    }
    const double2 lim = residual_limits(a, rec);
    uint8_t* keep = a.out.member_keep + off;
    const int32_t* mem = a.members + off;
    __syncwarp();  // the previous bin's readers of the stage are done
#pragma unroll 4
    for (int j = lane; j < cnt; j += 32) {
      keep[j] = 1;
      if (j < kAffineStage) stage[j] = pair_coords(a, mem, j);
    }
    __syncwarp();
    auto pair_of = [&](int j) -> float4 { return j < kAffineStage ? stage[j] : pair_coords(a, mem, j); };
    int alive = cnt, passes = 0, live = 0, singular = 0, on_edge = 0;
    double pu[3] = {0, 0, 0}, pv[3] = {0, 0, 0};
    while (true) {
      double sxx = 0, sxy = 0, sx = 0, syy = 0, sy = 0, sn = 0;
      double sxu = 0, syu = 0, su = 0, sxv = 0, syv = 0, sv = 0;
      for (int j = lane; j < cnt; j += 32) {
        if (!keep[j]) continue;
        const float4 c = pair_of(j);
        const double x = c.x, y = c.y, u = c.z, w = c.w;
        sxx += x * x; sxy += x * y; sx += x; syy += y * y; sy += y; sn += 1.0;
        sxu += x * u; syu += y * u; su += u; sxv += x * w; syv += y * w; sv += w;
      }
      sxx = warp_sum(sxx); sxy = warp_sum(sxy); sx = warp_sum(sx); syy = warp_sum(syy);
      sy = warp_sum(sy); sn = warp_sum(sn); sxu = warp_sum(sxu); syu = warp_sum(syu);
      su = warp_sum(su); sxv = warp_sum(sxv); syv = warp_sum(syv); sv = warp_sum(sv);
      const double ru[3] = {sxu, syu, su}, rv[3] = {sxv, syv, sv};
      singular |= solve_affine(sxx, sxy, sx, syy, sy, sn, ru, rv, pu, pv);
      int removed = 0;
      for (int j = lane; j < cnt; j += 32) {
        if (!keep[j]) continue;
        const float4 c = pair_of(j);
        const double du = fit_residual(pu[0], pu[1], pu[2], c.x, c.y, c.z);
        const double dv = fit_residual(pv[0], pv[1], pv[2], c.x, c.y, c.w);
        on_edge += residual_on_edge(du, dv, lim.x, lim.y) ? 1 : 0;
        if (du > lim.x || dv > lim.y) {
          keep[j] = 0;
          ++removed;
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) removed += __shfl_xor_sync(0xffffffffu, removed, o);
      __syncwarp();
      alive -= removed;
      ++passes;
      if (alive < a.affine_threshold) break;  // dropped from valid_bins after this pass
      if (removed == 0) { live = 1; break; }
      if (a.max_passes > 0 && passes >= a.max_passes) { live = 1; break; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) on_edge += __shfl_xor_sync(0xffffffffu, on_edge, o);
    if (lane == 0) write_bin_result(a, v, pu, pv, alive, live, singular, on_edge, passes);
   }
  }
}

// The Hough records of the bins that entered the affine stage, in the order of sod_affine_out.valid_bin:
// what a caller reads back next to params / votes / status (one coalesced copy instead of four gathers).
__global__ void valid_records_kernel(const int32_t* __restrict__ counters, const int32_t* __restrict__ valid_bin,
                                     int64_t cap_valid, const int32_t* __restrict__ bin_group,
                                     const int32_t* __restrict__ bin_code, const int64_t* __restrict__ bin_order,
                                     const double* __restrict__ bin_mean, int32_t* __restrict__ out_group,
                                     int32_t* __restrict__ out_code, int64_t* __restrict__ out_order,
                                     double* __restrict__ out_mean) {
  int64_t n = counters[0];
  if (n > cap_valid) n = cap_valid;
  for (int64_t v = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; v < n;
       v += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int rec = valid_bin[v];
    out_group[v] = bin_group[rec];
    out_code[v] = bin_code[rec];
    out_order[v] = bin_order[rec];
#pragma unroll
    for (int c = 0; c < 6; ++c) out_mean[v * 6 + c] = bin_mean[static_cast<int64_t>(rec) * 6 + c];
  }
}

// remove_outliers with caller-supplied parameters (AffineParameters.py:128-155).
__global__ void affine_residual_kernel(const float2* __restrict__ mxy, const float2* __restrict__ qxy,
                                       int64_t n, const double* __restrict__ p, double x_ref,
                                       double y_ref, uint8_t* __restrict__ keep) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double x = mxy[i].x, y = mxy[i].y;
  const double ua = __dadd_rn(__dadd_rn(__dmul_rn(p[0], x), __dmul_rn(p[1], y)), p[4]);
  const double va = __dadd_rn(__dadd_rn(__dmul_rn(p[2], x), __dmul_rn(p[3], y)), p[5]);
  keep[i] = !(fabs(ua - static_cast<double>(qxy[i].x)) > x_ref || fabs(va - static_cast<double>(qxy[i].y)) > y_ref);
}

}  // namespace
}  // namespace sod

using namespace sod;

extern "C" int sod_valid_bin_records(const sod_hough_out* hough, const sod_affine_out* affine, int32_t* out_group,
                                     int32_t* out_code, int64_t* out_order, double* out_mean,
                                     sod_stream_t stream) {
  SOD_CHECK_ARG(hough && affine && out_group && out_code && out_order && out_mean, "null pointer");
  SOD_CHECK_ARG(affine->counters && affine->valid_bin && hough->bin_group && hough->bin_code && hough->bin_order &&
                    hough->bin_mean,
                "null input array");
  const int sms = device_sm_count();
  if (sms <= 0) return SOD_ERR_CUDA;
  valid_records_kernel<<<sms * 2, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      affine->counters, affine->valid_bin, affine->cap_valid, hough->bin_group, hough->bin_code, hough->bin_order,
      hough->bin_mean, out_group, out_code, out_order, out_mean);
  SOD_CHECK_LAUNCH("valid_records_kernel");
  return SOD_OK;
}

extern "C" int sod_affine_residual_keep(const float* model_xy, const float* query_xy, int64_t n,
                                        const double* params, double x_ref, double y_ref,
                                        uint8_t* keep, sod_stream_t stream) {
  SOD_CHECK_ARG(n >= 0, "n < 0");
  if (n == 0) return SOD_OK;
  SOD_CHECK_ARG(model_xy && query_xy && params && keep, "null pointer");
  const int threads = 256;
  affine_residual_kernel<<<static_cast<unsigned>((n + threads - 1) / threads), threads, 0,
                           static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const float2*>(model_xy), reinterpret_cast<const float2*>(query_xy), n, params,
      x_ref, y_ref, keep);
  SOD_CHECK_LAUNCH("affine_residual_kernel");
  return SOD_OK;
}

extern "C" int sod_affine_verify(const sod_scene* scene, const int32_t* match_q, const int32_t* match_t,
                                 const sod_hough_out* hough, int32_t bins, int32_t vote_threshold,
                                 int32_t affine_threshold, double factor_x, double factor_y,
                                 int32_t max_passes, const sod_affine_out* out, sod_stream_t stream) {
  SOD_CHECK_ARG(scene && hough && out, "null scene/hough/out");
  SOD_CHECK_ARG(out->counters && out->valid_bin && out->params && out->votes && out->status &&
                    out->member_keep && out->cap_valid > 0 && out->cap_votes > 0,
                "null output array or zero capacity");
  SOD_CHECK_ARG(bins >= 1, "bins out of range");
  SOD_CHECK_ARG(match_q && match_t && hough->counters && hough->bin_group && hough->bin_code &&
                    hough->bin_count && hough->bin_offset && hough->members,
                "null input array");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  SOD_CHECK_CUDA(cudaMemsetAsync(out->counters, 0, 4 * sizeof(int32_t), st));
  const int sms = device_sm_count();
  if (sms <= 0) return SOD_ERR_CUDA;
  AffineArgs a;
  a.sc = *scene;
  a.match_q = match_q; a.match_t = match_t; a.hough_counters = hough->counters;
  a.bin_group = hough->bin_group; a.bin_code = hough->bin_code; a.bin_count = hough->bin_count;
  a.bin_offset = hough->bin_offset; a.members = hough->members; a.cap_bins = hough->cap_bins;
  a.bins = bins; a.vote_threshold = vote_threshold; a.affine_threshold = affine_threshold;
  a.factor_x = factor_x; a.factor_y = factor_y; a.max_passes = max_passes; a.out = *out;
  StageScope timed(SOD_STAGE_AFFINE, st);
  affine_select_kernel<<<sms * 4, 256, 0, st>>>(a);
  SOD_CHECK_LAUNCH("affine_select_kernel");
  affine_verify_small_kernel<<<sms * 5, kSmallThreads, 0, st>>>(a);  // 5 CTAs per SM are resident (registers)
  SOD_CHECK_LAUNCH("affine_verify_small_kernel");
  affine_verify_kernel<<<sms * 5, kAffineWarps * 32, 0, st>>>(a);
  SOD_CHECK_LAUNCH("affine_verify_kernel");
  return SOD_OK;
}
