// K0-K3: descriptor packing, database preparation, the tcgen05 2-NN matcher and the top-2 merge.
//
// Replaces cv2.BFMatcher().knnMatch(des_query, des, k=2) + the ratio loop of the reference
// (main.py:70-86).  |q-t|^2 = |q|^2 + |t|^2 - 2 q.t with u8 operands is exact in int32, so the
// contraction q.t runs on the 5th-gen tensor cores (tcgen05.mma kind::i8, u8 x u8 -> s32 in TMEM)
// and the top-2 selection happens in the TMEM epilogue without ever writing distances to HBM.
//
// Kernel anatomy (persistent CTA pairs: a cluster of 2 CTAs on the two SMs of a TPC, 640 threads each):
//   warp 0      TMA producer: the CTA's query block (4 x 128 rows, double buffered) + its half of each
//               database tile (64 of the tile's 128 rows = 8 KB, 8-deep ring) + the whole tile's 1040 B
//               slice of per-row constants (|t|^2 << 8 | column, chunk minima, original rows) in its own,
//               deeper ring.
//   warps 1, 3  MMA issuers of the leader CTA, two query tiles each (warp 1 -> tiles 0 and 2, warp 3 ->
//               tiles 1 and 3): per database tile and query tile 4 UTCIMMA.2CTA (M=256 over both CTAs,
//               N=128, K=32) into that query tile's 128-column TMEM accumulator slot (4 slots per CTA).
//   warp 2      TMEM allocator.
//   warps 4-19  epilogue: thread <-> query row (TMEM lane), 16 warps = 4 lane quadrants x 4 query tiles,
//               one thread per query row that sees every database tile.  A warp pulls the 128 columns of
//               its slot into registers in two loads, releases the slot, and prunes: a column can only
//               enter the row's top-2 if |t|^2 - 2 q.t <= current 2nd best.
//
// Pruning needs a bound that is tight PER ROW: a warp takes the slow path as soon as one of its 32
// rows does.  sod_db_prepare therefore stores the database sorted by |t|^2, so that the smallest
// |t|^2 of a 32-column chunk (cmin) is within a few units of every member and
//     cmin - 2 * max_j acc_j  >  2nd best      (one 3-input max tree on the raw accumulators)
// rejects almost every chunk after the first few thousand columns.  Inside a tile rows are ordered
// by original index and a permutation maps back, so results (incl. ties -> lowest original index,
// as cv2) do not depend on the reordering.
#include <climits>
#include <cub/device/device_radix_sort.cuh>

#include "sod_common.cuh"
#include "sod_ptx.cuh"
#include "sod_tma.cuh"
#include "sod_top2.cuh"

namespace sod {
namespace {

constexpr int kTileM = 128;                 // query rows per MMA (TMEM lanes)
constexpr int kQTiles = 4;                  // query tiles per CTA sharing one database tile
constexpr int kBlockQ = kTileM * kQTiles;   // 512 query rows per CTA (a pair unit sweeps 1024)
constexpr int kAbiBlockQ = 256;             // query block of the C ABI: row_thr is padded to it and
                                            // block_rotation counts it
constexpr int kTileN = SOD_TILE_ROWS;       // database rows per MMA
constexpr int kTileBytes = kTileN * SOD_DESC_DIM;  // 16 KB (A half-tile has the same size)
constexpr int kChunk = 32;                  // accumulator columns per tcgen05.ld
constexpr int kCqTile = SOD_CQ_TILE_INTS;   // 128 x |t|^2 + 4 per-chunk minima + 128 x original row
constexpr int kCqPerm = kTileN + 4;         // offset of the permutation inside a tile's slice
constexpr int kCqTileBytes = kCqTile * 4;   // 1040 B, a multiple of 16 for the bulk copy
constexpr int kNoKey = 0x7FFFFF;            // |t|^2 of padding rows / "no candidate yet" (> 128*255^2,
                                            // and (kNoKey << 8 | 127) still fits int32)
constexpr int kEpiWarps = 4 * kQTiles;      // (TMEM lane quadrant) x (query tile); one candidate list per
                                            // row and segment
constexpr int kIssuers = 2;                 // MMA-issuing warps (1 and 3), kQTiles / kIssuers tiles each
constexpr int kThreads = (4 + kEpiWarps) * 32;
constexpr int kTmemCols = 512;
constexpr int kRegsLight = 56;      // producer / MMA / allocator warpgroup after setmaxnreg.dec
constexpr int kRegsEpilogue = 104;  // 64 accumulators + keys + state
// setmaxnreg only moves registers inside the CTA's launch allocation (threads x launch registers,
// the latter a multiple of 8): asking for more makes setmaxnreg.inc wait forever.
constexpr int kRegsLaunch = 65536 / kThreads / 8 * 8;
static_assert(128 * kRegsLight + kEpiWarps * 32 * kRegsEpilogue <= kThreads * kRegsLaunch,
              "setmaxnreg budget exceeds the CTA's register pool");

static_assert(kQTiles * kTileN == kTmemCols, "one 128-column accumulator slot per query tile fills TMEM");

// Shared-memory layout.  A CTA holds HALF of every database tile (64 rows, 8 KB).
constexpr int kStages = 8;                   // database ring depth
constexpr int kBStageBytes = kTileBytes / 2;
constexpr int kCqSlots = 16;                 // >= kStages + 2 (slot-reuse argument in the producer);
                                             // a power of two keeps `step % slots` a mask
constexpr int kOffA = 0;                                     // [2 buffers][4 query tiles][16 KB]
constexpr int kOffB = kOffA + 2 * kQTiles * kTileBytes;      // [stages][8 KB]
constexpr int kOffCq = kOffB + kStages * kBStageBytes;       // [cq slots][260] int32
constexpr int kOffBar = kOffCq + kCqSlots * kCqTileBytes;
constexpr int kNumBars = 2 * kStages + 4 + 2 * kQTiles + kCqSlots;
constexpr int kOffTmemPtr = kOffBar + kNumBars * 8;
constexpr int kSmemBytes = kOffTmemPtr + 16 + 1024;          // +1024: manual 1 KB alignment
static_assert(kCqSlots >= kStages + 2 && (kCqSlots & (kCqSlots - 1)) == 0, "cq ring too shallow");
static_assert(kSmemBytes <= 227 * 1024, "shared memory exceeds the 227 KB a block may use");

struct MatchArgs {
  const int32_t* qn;   // [nq] |q|^2
  const int32_t* cq;   // [n_tiles][260] per stored row: |t|^2 << 8 | column, chunk minima of |t|^2,
                       // original row (-1 = padding)
  uint32_t* part_d2;   // [n_seg][nq][2]  (one list per segment)
  int32_t* part_idx;   // [n_seg][nq][2]
  int32_t* row_thr;    // [thr_rows] shared pruning thresholds (memset to 0x7F..), or nullptr
  int nq;
  int thr_rows;        // nq rounded up to kAbiBlockQ (sod_row_thr_ints): rows past it have no threshold
  int n_tiles;         // tiles swept by this launch: [tile_begin, tile_begin + n_tiles)
  int tile_begin;
  int n_qunits;        // units per segment: ceil(n_qblocks / 2), a CTA pair sweeps two query blocks (1024 rows)
  int n_seg;
  int idx_base;
  // Threshold publishing over peer memory (database sharded over several GPUs, kSeeded sweeps): when a unit
  // ends, the 2nd best of each of its rows is min-ed into EVERY rank's threshold array (own one included);
  // unit_rot rotates the order in which this rank visits the query blocks, so that the ranks reach a block at
  // different times and a later visitor prunes with what the earlier ones found in their shards.
  int n_peers;
  int unit_rot;
  int32_t* peer_thr[SOD_EXCHANGE_MAX_RANKS];
};

// 3-input max: top2_chunk builds a balanced tree (depth 4) over 32 registers with them; the
// serial form is a 16-deep dependent chain of VIMNMX3.
__device__ __forceinline__ int imax3(int a, int b, int c) { return max(max(a, b), c); }
// Running top-2 of one query row as two 64-bit keys (d << 32 | original index), d = d2 - |q|^2:
// signed 64-bit order is the (distance, index) lexicographic order.
struct Top2 {
  long long k1, k2;
  int d2;  // high word of k2: the pruning threshold
  __device__ __forceinline__ void offer(int d, int i) {
    const long long key = (static_cast<long long>(d) << 32) | static_cast<unsigned>(i);
    if (key < k1) {
      k2 = k1;
      k1 = key;
    } else if (key < k2) {
      k2 = key;
    }
    d2 = static_cast<int>(k2 >> 32);
  }
};
constexpr long long kNoKey64 = (static_cast<long long>(kNoKey) << 32) | 0x7FFFFFFF;

// One chunk of 32 accumulator columns, in levels of increasing cost:
//  1. bound: every element has |t|^2 - 2 q.t >= cmin - 2*max(acc); if that exceeds the row's 2nd
//     best nothing can change (~0.5 ALU op per element, tight because the database is norm-sorted);
//  2. the same bound per sub-tree of the max tree (9 + 9 + 9 + 5 elements, its maxima are already
//     there): only sub-trees that fail it are looked at;
//  3. inside those: the exact packed keys ((|t|^2 - 2 q.t) << 8 | tile column) by one IMAD each
//     from the prepared (|t|^2 << 8 | column) and a running (smallest, 2nd smallest) (columns inside
//     a tile are in original-index order, so ties inside the tile resolve correctly), then at most
//     two offers to the running best with the ORIGINAL row index read through the permutation in
//     shared memory, which settles ties across tiles exactly as cv2 does (lowest original index).
// The epilogue is bound by ALU issue slots, so the instruction count of this rare path matters: a
// branch-free 32-key tournament (+53 instructions) cost 5 %, finer sub-trees (more branches) 10 %.
// All tests are exact; pruning never changes the result.
// `thr` is the pruning threshold: the row's 2nd best over everything its thread has seen, and over what
// other units sweeping the row have published (an element above it cannot be in the merged top-2; ties
// go through).
__device__ __forceinline__ void top2_chunk(const uint32_t* v, const int4* __restrict__ cp4,
                                           int cmin, const int32_t* __restrict__ perm_s,
                                           int idx_base, Top2& best, int& thr) {
  // level 1, with the sub-tree maxima of the balanced tree kept: elements 0-8, 9-17, 18-26, 27-31
  const int* av = reinterpret_cast<const int*>(v);
  int t[11];
#pragma unroll
  for (int i = 0; i < 10; ++i) t[i] = imax3(av[3 * i], av[3 * i + 1], av[3 * i + 2]);
  t[10] = max(av[30], av[31]);
  const int u0 = imax3(t[0], t[1], t[2]), u1 = imax3(t[3], t[4], t[5]), u2 = imax3(t[6], t[7], t[8]);
  const int u3 = max(t[9], t[10]);
  if (cmin - 2 * max(imax3(u0, u1, u2), u3) > thr) return;
  // levels 2 + 3 only inside the sub-trees whose own bound fails: exact packed keys by one IMAD
  // each and a running (smallest, 2nd smallest)
  const int* cp = reinterpret_cast<const int*>(cp4);
  int t1 = INT_MAX, t2 = INT_MAX;
  auto scan = [&](int lo, int hi) {
#pragma unroll
    for (int j = lo; j < hi; ++j) {
      const int key = cp[j] - 512 * av[j];
      const int m = max(t1, key);
      t1 = min(t1, key);
      t2 = min(t2, m);
    }
  };
  if (cmin - 2 * u0 <= thr) scan(0, 9);
  if (cmin - 2 * u1 <= thr) scan(9, 18);
  if (cmin - 2 * u2 <= thr) scan(18, 27);
  if (cmin - 2 * u3 <= thr) scan(27, 32);
  if ((t1 >> 8) > thr) return;
  SOD_DCHECK((t1 & 0xFF) < kTileN && (t2 == INT_MAX || (t2 & 0xFF) < kTileN));
  const int o1 = perm_s[t1 & 0xFF];
  if (o1 >= 0) best.offer(t1 >> 8, idx_base + o1);
  thr = min(thr, best.d2);
  if ((t2 >> 8) <= thr) {
    const int o2 = perm_s[t2 & 0xFF];
    if (o2 >= 0) best.offer(t2 >> 8, idx_base + o2);
    thr = min(thr, best.d2);
  }
}

// kShare: query rows are swept by several units that share their thresholds through a.row_thr.
// kSeeded: a.row_thr is only read when a unit starts and updated once when it ends - for
// single-segment sweeps with caller-held thresholds (the seeded shard sweeps of a database-sharded
// run), which have nobody to share with inside the launch and must not pay the per-tile load and
// atomicMin of the sharing code (B200, 1.28 M queries x 125k-row shard: 15.27 ms against 16.21 ms
// with the sharing instance and 16.44 ms unseeded; profiles/r02_threshold_seeding.txt).
// The two CTAs of a cluster (the two SMs of a TPC) run ONE tcgen05.mma.cta_group::2 per query tile over
// M = 256 rows - 128 query rows of each CTA - and N = 128 database rows, of which each CTA stages 64: the
// database stream from L2 and the shared-memory operand reads per MAC are half of what one CTA per tile
// would need (B: 8 KB instead of 16 KB per CTA and tile).  The accumulators and the whole epilogue are per
// CTA.  The leader CTA (cluster rank 0) issues the MMAs; TMA loads of both CTAs report to the leader's
// "full" barriers, tcgen05.commit multicasts "free" / "accumulator ready" to both CTAs, and the epilogue
// warps of both CTAs release accumulator slots on the leader's barriers.
template <bool kShare, bool kSeeded = false>
__global__ void __launch_bounds__(kThreads, 1)
match_top2_kernel(const __grid_constant__ CUtensorMap tmap_q,
                  const __grid_constant__ CUtensorMap tmap_db, const MatchArgs a) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;  // SWIZZLE_128B tiles need 1 KB alignment
  uint8_t* smem = smem_raw + (base - raw_addr);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t cta_rank = cluster_ctarank();   // 0 = leader of the pair
  const int unit0 = static_cast<int>(cluster_id_x());
  const int unit_step = static_cast<int>(cluster_count_x());

  const uint32_t bar0 = base + kOffBar;
  auto bar_full = [&](int s) { return bar0 + 8u * s; };
  auto bar_empty = [&](int s) { return bar0 + 8u * (kStages + s); };
  auto bar_afull = [&](int b) { return bar0 + 8u * (2 * kStages + b); };
  auto bar_aempty = [&](int b) { return bar0 + 8u * (2 * kStages + 2 + b); };
  // accumulator hand-off barriers of query tile h's TMEM slot: one phase per tile step
  auto bar_tfull = [&](int h) { return bar0 + 8u * (2 * kStages + 4 + h); };
  auto bar_tempty = [&](int h) { return bar0 + 8u * (2 * kStages + 4 + kQTiles + h); };
  auto bar_cqfull = [&](int s) { return bar0 + 8u * (2 * kStages + 4 + 2 * kQTiles + s); };
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem + kOffTmemPtr);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_q);
    tma_prefetch_desc(&tmap_db);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(bar_full(s), 1);
      mbar_init(bar_empty(s), kIssuers);  // one tcgen05.commit per issuing warp
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(bar_afull(b), 1);
      mbar_init(bar_aempty(b), kIssuers);
    }
    for (int h = 0; h < kQTiles; ++h) {
      mbar_init(bar_tfull(h), 1);
      mbar_init(bar_tempty(h), 8);  // the four quadrant warps that read one slot, of each CTA
    }
    for (int s = 0; s < kCqSlots; ++s) mbar_init(bar_cqfull(s), 1);
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc_pair(smem_u32(const_cast<uint32_t*>(tmem_ptr_smem)), kTmemCols);
    tmem_relinquish_pair();
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  const int total_units = a.n_qunits * a.n_seg;

  if (warp < 4) {
    if constexpr (kRegsLight < kRegsLaunch)
      setmaxnreg_dec<kRegsLight>();  // this warpgroup hands its registers to the epilogue warpgroups
  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      uint32_t step = 0, ucount = 0;
      for (int u = unit0; u < total_units; u += unit_step, ++ucount) {
        const int seg = u / a.n_qunits;
        int qu = u - seg * a.n_qunits + a.unit_rot;   // unit_rot < n_qunits (0 unless n_seg == 1)
        if (qu >= a.n_qunits) qu -= a.n_qunits;
        const int qb = qu * 2 + static_cast<int>(cta_rank);
        const int t0 = a.tile_begin + static_cast<int>(static_cast<int64_t>(seg) * a.n_tiles / a.n_seg);
        const int t1 = a.tile_begin + static_cast<int>(static_cast<int64_t>(seg + 1) * a.n_tiles / a.n_seg);
        const uint32_t ab = ucount & 1u, aph = (ucount >> 1) & 1u;
        mbar_wait(bar_aempty(ab), aph ^ 1u);
        // both CTAs' query blocks report to the leader's barrier, which expects the bytes of both
        if (cta_rank == 0) mbar_arrive_expect_tx(bar_afull(ab), 2 * kQTiles * kTileBytes);
        const uint32_t afull_leader = mapa_shared(bar_afull(ab), 0);
        for (int h = 0; h < kQTiles; ++h)
          tma_load_2d_pair(base + kOffA + (ab * kQTiles + h) * kTileBytes, &tmap_q, afull_leader, 0,
                           qb * kBlockQ + h * kTileM);
        for (int t = t0; t < t1; ++t, ++step) {
          const uint32_t s = step % kStages, ph = (step / kStages) & 1u;
          mbar_wait(bar_empty(s), ph ^ 1u);
          // this CTA stages rows [64 * rank, 64 * rank + 64) of the tile
          if (cta_rank == 0) mbar_arrive_expect_tx(bar_full(s), 2 * kBStageBytes);
          tma_load_2d_pair(base + kOffB + s * kBStageBytes, &tmap_db, mapa_shared(bar_full(s), 0), 0,
                           t * kTileN + static_cast<int>(cta_rank) * (kTileN / 2));
          // cq slice rides in its own, deeper ring: stage s is released when the MMAs that read it
          // retire, but the epilogue still reads cq after it has handed the accumulator back.
          // The write for step j happens after the MMAs of step j-kStages (all four query tiles)
          // retired; each of them was issued after the epilogue warps of its tile RELEASED step
          // j-kStages-1, so every epilogue warp has finished its arithmetic on step j-kStages-2.
          // Steps j-kStages-1 .. j-1 may still be live -> kStages+2 = 10 of the 16 slots are needed.
          // Every CTA needs the constants of the WHOLE tile - its accumulators span all 128 database
          // rows - and loads them itself; the argument holds per CTA because the MMAs are joint.
          const uint32_t slot = step % kCqSlots;
          mbar_arrive_expect_tx(bar_cqfull(slot), kCqTileBytes);
          bulk_load_1d(base + kOffCq + slot * kCqTileBytes, a.cq + static_cast<int64_t>(t) * kCqTile,
                       kCqTileBytes, bar_cqfull(slot));
        }
      }
    }
  } else if ((warp == 1 || warp == 3) && cta_rank == 0) {
    // ------------------------------------------------------------------ MMA issuers
    // Two issuing warps with two query tiles each (warp 1 -> tiles 0 and 2, warp 3 -> tiles 1 and 3, so
    // that the tensor pipe sees the tiles of a stage roughly in the order 0, 1, 2, 3): with K = 128 an
    // accumulator slot holds only 256 clk of tensor work, so the issuing warp's own instruction stream
    // and barrier round trips must stay well below that per slot.  Slot h is reused at the next tile
    // step, after the MMAs of the three other query tiles (768 clk): that is the epilogue's window to
    // pull it into registers.  Each warp runs its loop convergently so that addresses, phases and
    // descriptors live in uniform registers; only the tcgen05 instructions are issued by one elected
    // lane.  (Inside a divergent `if (lane == 0)` every UTCIMMA operand needs an R2UR move.)
    const int h0 = warp >> 1;
    constexpr uint32_t idesc = umma_idesc_u8(2 * kTileM, kTileN);
    uint32_t step = 0, ucount = 0;
    for (int u = unit0; u < total_units; u += unit_step, ++ucount) {
      const int seg = u / a.n_qunits;
      const int t0 = a.tile_begin + static_cast<int>(static_cast<int64_t>(seg) * a.n_tiles / a.n_seg);
      const int t1 = a.tile_begin + static_cast<int>(static_cast<int64_t>(seg + 1) * a.n_tiles / a.n_seg);
      const uint32_t ab = ucount & 1u, aph = (ucount >> 1) & 1u;
      mbar_wait(bar_afull(ab), aph);
      const uint32_t a_buf = base + kOffA + ab * (kQTiles * kTileBytes);
      for (int t = t0; t < t1; ++t, ++step) {
        const uint32_t s = step % kStages, ph = (step / kStages) & 1u;
        const uint64_t bdesc = umma_desc_k128(base + kOffB + s * kBStageBytes);
        mbar_wait(bar_full(s), ph);
#pragma unroll
        for (int i = 0; i < kQTiles / kIssuers; ++i) {
          const int h = h0 + kIssuers * i;
          const uint64_t adesc = umma_desc_k128(a_buf + h * kTileBytes);
          if (step >= 1)  // slot h was last used by step - 1: wait for its epilogue warps' release
            mbar_wait(bar_tempty(h), (step - 1) & 1u);
          tc_fence_after();
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < SOD_DESC_DIM / 32; ++k)  // K = 32 bytes per UTCIMMA: +2 x 16 B
              umma_i8_pair(tmem_base + h * kTileN, adesc + 2 * k, bdesc + 2 * k, idesc, k > 0);
            umma_commit_pair(bar_tfull(h), 3);  // this query tile is ready in both CTAs
            // (count 2) stage free in both CTAs once both warps' tiles retire
            if (i == kQTiles / kIssuers - 1) umma_commit_pair(bar_empty(s), 3);
          }
          __syncwarp();
        }
      }
      if (elect_one()) umma_commit_pair(bar_aempty(ab), 3);  // (count 2) query block buffer free
      __syncwarp();
    }
  }
  } else {
    // ------------------------------------------------------------------ epilogue
    if constexpr (kRegsEpilogue > kRegsLaunch) setmaxnreg_inc<kRegsEpilogue>();
    const int e = warp - 4;
    const int quad = warp & 3;          // TMEM lane quadrant this warp may read
    const int h = e >> 2;               // which query tile
    const uint32_t lane_sel = static_cast<uint32_t>(quad * 32) << 16;
    // Loop invariants the compiler would otherwise rebuild at the top of EVERY tile step from special
    // registers (S2R SR_TID.X for the query tile, S2R SR_CgaCtaId for the shared-memory window of a cluster
    // launch - tens of cycles each, in front of the barrier waits): keep them in registers.
    uint32_t tfull_h = bar_tfull(h);
    uint32_t cqfull_0 = bar_cqfull(0);       // + 8 * slot
    uint32_t cq_0 = base + kOffCq;           // + slot * kCqTileBytes (shared-memory window address)
    uint32_t taddr = tmem_base + lane_sel + h * kTileN;     // this warp's lanes of slot h
    asm volatile("" : "+r"(tfull_h), "+r"(cqfull_0), "+r"(taddr), "+r"(cq_0));
    // accumulator slots are released on the LEADER's barriers (the leader issues the MMAs); kept in a
    // register: rematerialised, each release would re-read the cluster rank (S2R, tens of cycles) on the
    // critical path between the TMEM load and the slot's release
    uint32_t tempty_rel = mapa_shared(bar_tempty(h), 0);
    asm volatile("" : "+r"(tempty_rel));
    uint32_t step = 0, ucount = 1;
    for (int u = unit0; u < total_units; u += unit_step, ++ucount) {
      const int seg = u / a.n_qunits;
      int qu = u - seg * a.n_qunits + a.unit_rot;
      if (qu >= a.n_qunits) qu -= a.n_qunits;
      const int qb = qu * 2 + static_cast<int>(cta_rank);
      const int t0 = a.tile_begin + static_cast<int>(static_cast<int64_t>(seg) * a.n_tiles / a.n_seg);
      const int t1 = a.tile_begin + static_cast<int>(static_cast<int64_t>(seg + 1) * a.n_tiles / a.n_seg);
      const int row = qb * kBlockQ + h * kTileM + quad * 32 + lane;
      Top2 best{kNoKey64, kNoKey64, kNoKey};
      // Threshold sharing between the units that sweep different database segments for the same
      // query rows: every holder of the row publishes its 2nd best with atomicMin, everyone prunes
      // with the minimum.  Any unit's 2nd best is an upper bound of the row's final 2nd best, so this
      // stays exact; without it every segment pays the ~2 ln(n) threshold-establishing updates again.  (row_thr is padded to 256 rows; the rest of the
      // last query block, and the phantom block of an odd pair, lie past it and are never read or written.)
      const bool thr_row = (kShare || kSeeded) && row < a.thr_rows;
      int* const gthr = (kShare || kSeeded) ? a.row_thr + row : nullptr;
      int published = kNoKey;
      int thr = thr_row ? min(kNoKey, __ldcg(gthr)) : kNoKey;
      const uint32_t step_end = step + static_cast<uint32_t>(t1 - t0);
      for (; step < step_end; ++step) {
        const uint32_t slot = step % kCqSlots, cqph = (step / kCqSlots) & 1u;
        mbar_wait(cqfull_0 + 8u * slot, cqph);  // landed long ago: returns at the first poll
        mbar_wait(tfull_h, step & 1u);
        tc_fence_after();
        const int32_t* cs = reinterpret_cast<const int32_t*>(__cvta_shared_to_generic(cq_0 + slot * kCqTileBytes));
        const int32_t* perm_s = cs + kCqPerm;
        // fetched now, folded in after this tile: the L2 round trip hides behind the tile's work
        const int g_next = (kShare && thr_row) ? __ldcg(gthr) : kNoKey;
        const int4* c4 = reinterpret_cast<const int4*>(cs);
        const int4 cmin = c4[kTileN / 4];
        uint32_t v[2 * kChunk];
        tmem_ld64_wait(taddr, v);
        top2_chunk(v, c4, cmin.x, perm_s, a.idx_base, best, thr);
        top2_chunk(v + kChunk, c4 + 8, cmin.y, perm_s, a.idx_base, best, thr);
        tmem_ld64_wait(taddr + 2 * kChunk, v);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(tempty_rel);
        top2_chunk(v, c4 + 16, cmin.z, perm_s, a.idx_base, best, thr);
        top2_chunk(v + kChunk, c4 + 24, cmin.w, perm_s, a.idx_base, best, thr);
        if (kShare && thr_row) {
          if (best.d2 < published) {
            published = best.d2;
            atomicMin(gthr, published);
          }
          thr = min(thr, g_next);
        }
      }
      if (kSeeded && thr_row && best.d2 < kNoKey) {
        if (a.n_peers > 0) {
          // reductions over NVLink into every rank's array (no return value: fire and forget)
          const int64_t slot = gthr - a.row_thr;
          for (int p = 0; p < a.n_peers; ++p) atomicMin(a.peer_thr[p] + slot, best.d2);
        } else {
          atomicMin(gthr, best.d2);
        }
      }
      if (row < a.nq) {
        const int qn = a.qn[row];
        const int64_t o = (static_cast<int64_t>(seg) * a.nq + row) * 2;
        SOD_DCHECK(seg < a.n_seg && (best.k1 == kNoKey64 || static_cast<int>(best.k1 & 0xFFFFFFFFll) >= a.idx_base));
        const int d1 = static_cast<int>(best.k1 >> 32), d2 = static_cast<int>(best.k2 >> 32);
        a.part_d2[o + 0] = d1 != kNoKey ? static_cast<uint32_t>(d1 + qn) : 0xFFFFFFFFu;
        a.part_d2[o + 1] = d2 != kNoKey ? static_cast<uint32_t>(d2 + qn) : 0xFFFFFFFFu;
        a.part_idx[o + 0] = d1 != kNoKey ? static_cast<int>(best.k1 & 0xFFFFFFFFll) : -1;
        a.part_idx[o + 1] = d2 != kNoKey ? static_cast<int>(best.k2 & 0xFFFFFFFFll) : -1;
      }
    }
  }

  tc_fence_before();
  cluster_sync_all();  // the peer's shared memory and barriers stay alive until both CTAs are done
  if (warp == 2) tmem_dealloc_pair(tmem_base, kTmemCols);
}

// ------------------------------------------------------------------------------------------------
// K1 (query side): eight threads per descriptor row, 16 bytes per thread (four rows per warp), __dp4a for
// the squares, a three-step shuffle inside the group of eight.  Streaming: 128 B in, 4 B out per row.
__global__ void row_sqnorm_kernel(const uint8_t* __restrict__ x, int64_t n_rows,
                                  int32_t* __restrict__ out) {
  const int64_t t = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t row = t >> 3;
  const int part = threadIdx.x & 7;
  uint32_t s = 0;
  if (row < n_rows) {
    const uint4 w = __ldg(reinterpret_cast<const uint4*>(x + row * SOD_DESC_DIM) + part);
    s = __dp4a(w.x, w.x, s);
    s = __dp4a(w.y, w.y, s);
    s = __dp4a(w.z, w.z, s);
    s = __dp4a(w.w, w.w, s);
  }
#pragma unroll
  for (int o = 4; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (part == 0 && row < n_rows) out[row] = static_cast<int32_t>(s);
}

// K1 (database side), step 1: |t|^2 of every row as a sort key, row index as the value.
__global__ void db_norm_kernel(const uint8_t* __restrict__ db, int64_t n_rows,
                               uint32_t* __restrict__ keys, int32_t* __restrict__ vals) {
  const int64_t row = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (row >= n_rows) return;
  const uint4* p = reinterpret_cast<const uint4*>(db + row * SOD_DESC_DIM);
  uint32_t s = 0;
#pragma unroll
  for (int j = 0; j < SOD_DESC_DIM / 16; ++j) {
    const uint4 w = __ldg(p + j);
    s = __dp4a(w.x, w.x, s);
    s = __dp4a(w.y, w.y, s);
    s = __dp4a(w.z, w.z, s);
    s = __dp4a(w.w, w.w, s);
  }
  keys[row] = s;
  vals[row] = static_cast<int32_t>(row);
}

// K1 step 3 (after the radix sort by |t|^2): one CTA per tile of 128 sorted rows.  Inside the tile
// the rows are re-ordered by original index (bitonic sort in shared memory; padding sorts last),
// then the tile's constants, permutation and descriptor rows are written.
__global__ void __launch_bounds__(kTileN)
db_tile_kernel(const uint8_t* __restrict__ db, int64_t n_rows, int64_t n_tiles, int64_t stride,
               const uint32_t* __restrict__ keys, const int32_t* __restrict__ vals,
               uint8_t* __restrict__ db_sorted, int32_t* __restrict__ cq) {
  __shared__ int s_idx[kTileN];
  __shared__ int s_c[kTileN];
  // Storage tile `tile` holds the tile of norm rank (tile * stride) mod n_tiles, stride coprime to
  // n_tiles: a sweep in storage order then samples the norm range evenly instead of ascending
  // (ascending order would make every tile improve the running minimum - the worst case for pruning).
  const int64_t tile = blockIdx.x;
  const int64_t rank = (tile * stride) % n_tiles;
  const int col = threadIdx.x;
  const int64_t src_pos = rank * kTileN + col;
  const int64_t pos = tile * kTileN + col;
  s_idx[col] = src_pos < n_rows ? vals[src_pos] : INT_MAX;
  s_c[col] = src_pos < n_rows ? static_cast<int>(keys[src_pos]) : kNoKey;
  __syncthreads();
  for (int k = 2; k <= kTileN; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      const int partner = col ^ j;
      if (partner > col) {
        const bool up = (col & k) == 0;
        const int a = s_idx[col], b = s_idx[partner];
        if ((a > b) == up) {
          s_idx[col] = b; s_idx[partner] = a;
          const int ca = s_c[col];
          s_c[col] = s_c[partner]; s_c[partner] = ca;
        }
      }
      __syncthreads();
    }
  }
  const int idx = s_idx[col];
  const int c = s_c[col];
  int32_t* out = cq + tile * kCqTile;
  out[col] = (c << 8) | col;  // packed key base; padding rows: (kNoKey << 8 | col), never selected
  out[kCqPerm + col] = idx == INT_MAX ? -1 : idx;
  int cm = c;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cm = min(cm, __shfl_xor_sync(0xffffffffu, cm, o));
  if ((col & 31) == 0) out[kTileN + (col >> 5)] = cm;
  uint4* dst = reinterpret_cast<uint4*>(db_sorted + pos * SOD_DESC_DIM);
  if (idx != INT_MAX) {
    const uint4* src = reinterpret_cast<const uint4*>(db + static_cast<int64_t>(idx) * SOD_DESC_DIM);
#pragma unroll
    for (int j = 0; j < SOD_DESC_DIM / 16; ++j) dst[j] = __ldg(src + j);
  } else {
#pragma unroll
    for (int j = 0; j < SOD_DESC_DIM / 16; ++j) dst[j] = make_uint4(0, 0, 0, 0);  // padding row
  }
}

struct PrepWs {
  uint32_t *keys_in, *keys_out;
  int32_t *vals_in, *vals_out;
  void* cub_temp;
  size_t cub_bytes, bytes;
};

PrepWs carve_prep_ws(void* base, int64_t n) {
  PrepWs w;
  size_t o = 0;
  auto take = [&](size_t bytes) {
    void* p = base ? static_cast<char*>(base) + o : nullptr;
    o += (bytes + 255) & ~static_cast<size_t>(255);
    return p;
  };
  w.keys_in = static_cast<uint32_t*>(take(n * 4));
  w.keys_out = static_cast<uint32_t*>(take(n * 4));
  w.vals_in = static_cast<int32_t*>(take(n * 4));
  w.vals_out = static_cast<int32_t*>(take(n * 4));
  w.cub_bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, w.cub_bytes, w.keys_in, w.keys_out, w.vals_in, w.vals_out,
                                  static_cast<int>(n), 0, 24);
  w.cub_temp = take(w.cub_bytes);
  w.bytes = o;
  return w;
}

// K0: float32 -> u8 with an integrality check.
__global__ void pack_u8_kernel(const float4* __restrict__ src, int64_t n_vec4,
                               uchar4* __restrict__ dst, int32_t* __restrict__ nonint_flag) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n_vec4) return;
  const float4 f = src[i];
  const float r[4] = {f.x, f.y, f.z, f.w};
  unsigned char b[4];
  bool bad = false;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float c = fminf(fmaxf(r[k], 0.f), 255.f);
    const float q = rintf(c);
    bad |= !(q == r[k]);
    b[k] = static_cast<unsigned char>(q);
  }
  dst[i] = make_uchar4(b[0], b[1], b[2], b[3]);
  if (bad) atomicOr(nonint_flag, 1);
}

// K3: merge candidate lists, exact ratio test.
__global__ void top2_merge_kernel(const int32_t* __restrict__ parts_idx,
                                  const uint32_t* __restrict__ parts_d2, int n_parts, int64_t nq,
                                  int32_t* __restrict__ out_idx, uint32_t* __restrict__ out_d2,
                                  float* __restrict__ out_dist, uint8_t* __restrict__ out_pass,
                                  double ratio) {
  const int64_t row = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (row >= nq) return;
  uint32_t d1 = 0xFFFFFFFFu, d2 = 0xFFFFFFFFu;
  int32_t i1 = -1, i2 = -1;
  for (int p = 0; p < n_parts; ++p) {
    const int64_t o = (static_cast<int64_t>(p) * nq + row) * 2;
    const int2 ci = *reinterpret_cast<const int2*>(parts_idx + o);
    const uint2 cd = *reinterpret_cast<const uint2*>(parts_d2 + o);
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int32_t ci_j = j ? ci.y : ci.x;
      const uint32_t cd_j = j ? cd.y : cd.x;
      if (ci_j < 0) continue;
      const bool lt1 = i1 < 0 || cd_j < d1 || (cd_j == d1 && ci_j < i1);
      const bool lt2 = i2 < 0 || cd_j < d2 || (cd_j == d2 && ci_j < i2);
      if (lt1) {
        d2 = d1; i2 = i1;
        d1 = cd_j; i1 = ci_j;
      } else if (lt2) {
        d2 = cd_j; i2 = ci_j;
      }
    }
  }
  write_top2_row(row, i1, d1, i2, d2, out_idx, out_d2, out_dist, out_pass, ratio);
}

// K3, exchange form: candidate lists as packed keys (sod_top2.cuh).  Keys travel as [row][2] pairs, so a
// contiguous range of query rows is a contiguous message.
__global__ void top2_keys_kernel(const int32_t* __restrict__ idx, const uint32_t* __restrict__ d2, int64_t nq,
                                 int64_t n_rows, longlong2* __restrict__ keys) {
  const int64_t row = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (row >= n_rows) return;
  longlong2 k = make_longlong2(kNoneKey, kNoneKey);  // rows past nq: padding up to a whole number of slices
  if (row < nq)
    k = top2_pack_keys(*reinterpret_cast<const int2*>(idx + row * 2), *reinterpret_cast<const uint2*>(d2 + row * 2));
  keys[row] = k;
}

// n_parts lists of key pairs for the same rows -> the two smallest keys per row (keys of different
// database rows differ, so there is nothing to de-duplicate).
__global__ void top2_merge_keys_kernel(const longlong2* __restrict__ parts, int n_parts, int64_t n_rows,
                                       longlong2* __restrict__ out) {
  const int64_t row = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (row >= n_rows) return;
  long long k1 = kNoneKey, k2 = kNoneKey;
  for (int p = 0; p < n_parts; ++p) top2_fold_keys(k1, k2, parts[static_cast<int64_t>(p) * n_rows + row]);
  out[row] = make_longlong2(k1, k2);
}

__global__ void top2_from_keys_kernel(const longlong2* __restrict__ keys, int64_t nq,
                                      int32_t* __restrict__ out_idx, uint32_t* __restrict__ out_d2,
                                      float* __restrict__ out_dist, uint8_t* __restrict__ out_pass, double ratio) {
  const int64_t row = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (row >= nq) return;
  const longlong2 k = keys[row];
  write_top2_keys_row(row, k.x, k.y, out_idx, out_d2, out_dist, out_pass, ratio);
}

struct Plan {
  int n_tiles, n_qblocks, n_qunits, n_seg, grid;
};

// Per-unit cost outside its tile steps, in tile steps: the 12 steps of 2 query tiles measured for the earlier
// two-tile form, as time, in the twice-as-long steps of 4 query tiles (B200: 0.65 us against 0.36 us per step).
// A one-wave sweep timed at 64 .. 2048 tiles does not isolate it (the slow path is front-loaded, so the cost
// per step falls along the sweep); profiles/r04_match_four_tiles.txt.
constexpr int kUnitFillSteps = 6;

// Split every query block's database sweep into n_seg contiguous segments so that
// n_qunits*n_seg units fill the persistent grid evenly (cost = makespan in tile steps).  A unit is swept
// by a CTA pair (two query blocks of 512 rows side by side); the grid holds sms / 2 pairs (sms >= 2).
Plan make_plan(int64_t nq, int64_t ndb, int sms) {
  Plan p;
  p.n_tiles = static_cast<int>((ndb + kTileN - 1) / kTileN);
  p.n_qblocks = static_cast<int>((nq + kBlockQ - 1) / kBlockQ);
  p.n_qunits = (p.n_qblocks + 1) / 2;
  const int pairs = sms / 2;
  p.n_seg = 1;
  if (p.n_tiles > 0 && p.n_qblocks > 0) {
    const int max_seg = p.n_tiles < 512 ? p.n_tiles : 512;
    int64_t best = -1;
    for (int s = 1; s <= max_seg; ++s) {
      const int64_t units = static_cast<int64_t>(p.n_qunits) * s;
      const int64_t waves = (units + pairs - 1) / pairs;
      // + kUnitFillSteps: pipeline fill and the slow-path chunks of a unit's first columns (units of one
      // query block share their thresholds, so a later segment does not start from scratch)
      const int64_t cost = waves * ((p.n_tiles + s - 1) / s + kUnitFillSteps);
      if (best < 0 || cost < best) {
        best = cost;
        p.n_seg = s;
      }
    }
  }
  const int64_t units = static_cast<int64_t>(p.n_qunits) * p.n_seg;
  p.grid = static_cast<int>(units < pairs ? units : pairs) * 2;
  return p;
}

// [n_rows,128] u8 row-major, boxes of box_rows x 128 B, 128-byte swizzle, OOB rows read as zero.
int make_desc_map(CUtensorMap* m, const uint8_t* ptr, int64_t n_rows, int box_rows = kTileN) {
  return make_rowmajor_map(m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, ptr, n_rows, SOD_DESC_DIM, SOD_DESC_DIM,
                           box_rows);
}

}  // namespace
}  // namespace sod

using namespace sod;

extern "C" {

int64_t sod_cq_ints(int64_t n_rows) {
  return n_rows <= 0 ? 0 : (n_rows + kTileN - 1) / kTileN * kCqTile;
}

int sod_pack_u8_from_f32(const float* src, int64_t n_rows, uint8_t* dst, int32_t* nonint_flag,
                         sod_stream_t stream) {
  SOD_CHECK_ARG(n_rows >= 0, "n_rows < 0");
  if (n_rows == 0) return SOD_OK;
  SOD_CHECK_ARG(src && dst && nonint_flag, "null pointer");
  const int64_t n4 = n_rows * (SOD_DESC_DIM / 4);
  const int threads = 256;
  pack_u8_kernel<<<static_cast<unsigned>((n4 + threads - 1) / threads), threads, 0,
                   static_cast<cudaStream_t>(stream)>>>(reinterpret_cast<const float4*>(src), n4,
                                                        reinterpret_cast<uchar4*>(dst), nonint_flag);
  SOD_CHECK_LAUNCH("pack_u8_kernel");
  return SOD_OK;
}

size_t sod_db_prepare_workspace_bytes(int64_t n_rows) {
  if (n_rows <= 0) return 256;
  return carve_prep_ws(nullptr, n_rows).bytes + 256;
}

int sod_db_prepare(const uint8_t* db, int64_t n_rows, uint8_t* db_sorted, int32_t* cq, void* workspace,
                   size_t workspace_bytes, sod_stream_t stream) {
  SOD_CHECK_ARG(n_rows >= 0 && n_rows < (int64_t(1) << 31) - kTileN, "n_rows out of range");
  if (n_rows == 0) return SOD_OK;
  SOD_CHECK_ARG(db && db_sorted && cq && workspace, "null pointer");
  SOD_CHECK_ARG(db != db_sorted, "db_sorted must not alias db");
  SOD_CHECK_ARG((reinterpret_cast<uintptr_t>(db) & 15) == 0 && (reinterpret_cast<uintptr_t>(db_sorted) & 15) == 0 &&
                    (reinterpret_cast<uintptr_t>(workspace) & 255) == 0,
                "db/db_sorted must be 16-byte and workspace 256-byte aligned");
  PrepWs w = carve_prep_ws(workspace, n_rows);
  SOD_CHECK_ARG(workspace_bytes >= w.bytes, "workspace too small: %zu < %zu", workspace_bytes, w.bytes);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int threads = 128;
  db_norm_kernel<<<static_cast<unsigned>((n_rows + threads - 1) / threads), threads, 0, st>>>(
      db, n_rows, w.keys_in, w.vals_in);
  SOD_CHECK_LAUNCH("db_norm_kernel");
  // |t|^2 <= 128*255^2 < 2^24; LSD radix sort is stable, so equal norms stay in index order.
  SOD_CHECK_CUDA(cub::DeviceRadixSort::SortPairs(w.cub_temp, w.cub_bytes, w.keys_in, w.keys_out, w.vals_in,
                                                 w.vals_out, static_cast<int>(n_rows), 0, 24, st));
  const int64_t tiles = (n_rows + kTileN - 1) / kTileN;
  int64_t stride = static_cast<int64_t>(0.6180339887498949 * static_cast<double>(tiles)) | 1;
  auto gcd = [](int64_t a, int64_t b) { while (b) { const int64_t t = a % b; a = b; b = t; } return a; };
  while (gcd(stride, tiles) != 1) stride += 2;
  db_tile_kernel<<<static_cast<unsigned>(tiles), kTileN, 0, st>>>(db, n_rows, tiles, stride, w.keys_out,
                                                                 w.vals_out, db_sorted, cq);
  SOD_CHECK_LAUNCH("db_tile_kernel");
  return SOD_OK;
}

int sod_query_prepare(const uint8_t* q, int64_t n_rows, int32_t* qn, sod_stream_t stream) {
  SOD_CHECK_ARG(n_rows >= 0 && n_rows < (int64_t(1) << 31) - kBlockQ, "n_rows out of range");
  if (n_rows == 0) return SOD_OK;
  SOD_CHECK_ARG(q && qn, "null pointer");
  const int threads = 256;
  const int64_t blocks = (n_rows * 8 + threads - 1) / threads;
  row_sqnorm_kernel<<<static_cast<unsigned>(blocks), threads, 0, static_cast<cudaStream_t>(stream)>>>(
      q, n_rows, qn);
  SOD_CHECK_LAUNCH("row_sqnorm_kernel");
  return SOD_OK;
}

static int64_t thr_rows(int64_t n_query) {
  return n_query <= 0 ? 0 : (n_query + kAbiBlockQ - 1) / kAbiBlockQ * kAbiBlockQ;
}
// partial lists [n_seg][nq][2] (d2 + idx), then the shared thresholds [thr_rows(nq)]
static size_t match_lists_bytes(const Plan& p, int64_t n_query) {
  return static_cast<size_t>(p.n_seg) * static_cast<size_t>(n_query) * 2 * 8;
}
static size_t match_workspace_need(const Plan& p, int64_t n_query) {
  return match_lists_bytes(p, n_query) + static_cast<size_t>(thr_rows(n_query)) * 4;
}

int64_t sod_row_thr_ints(int64_t n_query) { return thr_rows(n_query); }

size_t sod_match_workspace_bytes(int64_t n_query, int64_t n_db) {
  if (n_query <= 0 || n_db <= 0) return 16;
  const int sms = device_sm_count();
  // (a device with fewer than two SMs is rejected by the match itself)
  return match_workspace_need(make_plan(n_query, n_db, sms >= 2 ? sms : 148), n_query) + 16;
}

int sod_match_top2(const uint8_t* q, const int32_t* qn, int64_t n_query, const uint8_t* db_sorted,
                   const int32_t* cq, int64_t n_db, int32_t db_index_base, int32_t* out_idx,
                   uint32_t* out_d2, void* workspace, size_t workspace_bytes, sod_stream_t stream) {
  return sod_match_top2_range(q, qn, n_query, db_sorted, cq, n_db, db_index_base, 0, -1, nullptr, out_idx, out_d2,
                              workspace, workspace_bytes, stream);
}

int sod_match_top2_range(const uint8_t* q, const int32_t* qn, int64_t n_query, const uint8_t* db_sorted,
                         const int32_t* cq, int64_t n_db, int32_t db_index_base, int64_t tile_begin,
                         int64_t tile_end, int32_t* row_thr, int32_t* out_idx, uint32_t* out_d2,
                         void* workspace, size_t workspace_bytes, sod_stream_t stream) {
  return sod_match_top2_peer(q, qn, n_query, db_sorted, cq, n_db, db_index_base, tile_begin, tile_end, row_thr, nullptr, 0,
                             0, out_idx, out_d2, workspace, workspace_bytes, stream);
}

int sod_match_top2_peer(const uint8_t* q, const int32_t* qn, int64_t n_query, const uint8_t* db_sorted,
                        const int32_t* cq, int64_t n_db, int32_t db_index_base, int64_t tile_begin,
                        int64_t tile_end, int32_t* row_thr, int32_t* const* peer_thr_host, int32_t n_peers,
                        int64_t block_rotation, int32_t* out_idx, uint32_t* out_d2, void* workspace,
                        size_t workspace_bytes, sod_stream_t stream) {
  SOD_CHECK_ARG(n_peers >= 0 && n_peers <= SOD_EXCHANGE_MAX_RANKS && (n_peers == 0 || (peer_thr_host && row_thr)),
                "bad peer threshold table");
  SOD_CHECK_ARG(block_rotation >= 0, "negative block rotation");
  SOD_CHECK_ARG(n_query >= 0 && n_db >= 0, "negative size");
  SOD_CHECK_ARG(n_query < (int64_t(1) << 31) - 2 * kBlockQ && n_db < (int64_t(1) << 31) - kTileN,
                "size out of range");
  SOD_CHECK_ARG(static_cast<int64_t>(db_index_base) + n_db < (int64_t(1) << 31),
                "db_index_base + n_db overflows int32");
  if (n_query == 0) return SOD_OK;
  SOD_CHECK_ARG(out_idx && out_d2, "null output pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int mthreads = 128;
  const unsigned mblocks = static_cast<unsigned>((n_query + mthreads - 1) / mthreads);
  const int64_t all_tiles = (n_db + kTileN - 1) / kTileN;
  if (tile_end < 0) tile_end = all_tiles;
  SOD_CHECK_ARG(tile_begin >= 0 && tile_begin <= tile_end && tile_end <= all_tiles, "tile range out of bounds");
  if (n_db == 0 || tile_begin == tile_end) {
    top2_merge_kernel<<<mblocks, mthreads, 0, st>>>(nullptr, nullptr, 0, n_query, out_idx, out_d2,
                                                    nullptr, nullptr, 0.0);
    SOD_CHECK_LAUNCH("top2_merge_kernel");
    return SOD_OK;
  }
  const uint8_t* db = db_sorted;
  SOD_CHECK_ARG(q && qn && db && cq && workspace, "null pointer");
  SOD_CHECK_ARG((reinterpret_cast<uintptr_t>(q) & 15) == 0 && (reinterpret_cast<uintptr_t>(db) & 15) == 0 &&
                    (reinterpret_cast<uintptr_t>(cq) & 15) == 0 &&
                    (reinterpret_cast<uintptr_t>(workspace) & 15) == 0,
                "q, db, cq and workspace must be 16-byte aligned");
  const int sms = device_sm_count();
  if (sms <= 0) return SOD_ERR_CUDA;
  if (sms < 2) {
    set_error("sod_match_top2: the matcher runs on CTA pairs and needs at least 2 SMs, the device has %d", sms);
    return SOD_ERR_UNSUPPORTED;
  }
  const Plan p = make_plan(n_query, (tile_end - tile_begin) * kTileN, sms);
  const size_t need = match_workspace_need(p, n_query);
  SOD_CHECK_ARG(workspace_bytes >= need, "workspace too small: %zu < %zu", workspace_bytes, need);

  CUtensorMap map_q, map_db;
  int rc = make_desc_map(&map_q, q, n_query);
  if (rc != SOD_OK) return rc;
  // stored padded to whole tiles; a CTA of a pair stages half a tile (64 rows) per step
  rc = make_desc_map(&map_db, db, (n_db + kTileN - 1) / kTileN * kTileN, kTileN / 2);
  if (rc != SOD_OK) return rc;

  MatchArgs a;
  a.qn = qn;
  a.cq = cq;
  a.part_d2 = static_cast<uint32_t*>(workspace);
  a.part_idx = reinterpret_cast<int32_t*>(a.part_d2 + static_cast<size_t>(p.n_seg) * n_query * 2);
  // Thresholds are shared whenever a query row is swept by more than one unit; 0x7F7F7F7F = none yet
  // A caller-held array additionally carries thresholds across launches (and, after a min-reduce, across
  // the shards of several GPUs): it is read at the start and holds min(input, this sweep's 2nd best) after.
  a.row_thr = row_thr;
  if (!row_thr && p.n_seg > 1) {
    a.row_thr = reinterpret_cast<int32_t*>(static_cast<uint8_t*>(workspace) + match_lists_bytes(p, n_query));
    SOD_CHECK_CUDA(cudaMemsetAsync(a.row_thr, 0x7F, static_cast<size_t>(thr_rows(n_query)) * 4, st));
  }
  a.nq = static_cast<int>(n_query);
  a.thr_rows = static_cast<int>(thr_rows(n_query));
  a.n_tiles = p.n_tiles;
  a.tile_begin = static_cast<int>(tile_begin);
  a.n_qunits = p.n_qunits;
  a.n_seg = p.n_seg;
  a.idx_base = db_index_base;
  // peer publishing and the rotated visiting order belong to single-segment sweeps (the seeded instance)
  const bool peer_mode = n_peers > 0 && row_thr && p.n_seg == 1;
  a.n_peers = peer_mode ? n_peers : 0;
  // block_rotation counts blocks of 256 query rows; a unit holds 2 * kBlockQ = 1024
  a.unit_rot = peer_mode ? static_cast<int>((block_rotation / (2 * kBlockQ / kAbiBlockQ)) % p.n_qunits) : 0;
  for (int i = 0; i < SOD_EXCHANGE_MAX_RANKS; ++i) a.peer_thr[i] = (peer_mode && i < n_peers) ? peer_thr_host[i] : nullptr;
  for (int i = 0; i < a.n_peers; ++i) SOD_CHECK_ARG(a.peer_thr[i], "null threshold array of rank %d", i);

  // The attribute is per device (a process may drive several), so it is set at every launch: ~1 us.
  const bool seeded = row_thr && p.n_seg == 1, share = a.row_thr && !seeded;
  auto* kernel = seeded ? match_top2_kernel<false, true>
                        : share ? match_top2_kernel<true, false> : match_top2_kernel<false, false>;
  SOD_CHECK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
  {
    StageScope timed(SOD_STAGE_MATCH, st);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(static_cast<unsigned>(p.grid));
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = static_cast<size_t>(kSmemBytes);
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    SOD_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kernel, map_q, map_db, a));
  }
  SOD_CHECK_LAUNCH("match_top2_kernel");
  top2_merge_kernel<<<mblocks, mthreads, 0, st>>>(a.part_idx, a.part_d2, p.n_seg, n_query,
                                                  out_idx, out_d2, nullptr, nullptr, 0.0);
  SOD_CHECK_LAUNCH("top2_merge_kernel");
  return SOD_OK;
}

int sod_top2_merge(const int32_t* parts_idx, const uint32_t* parts_d2, int32_t n_parts,
                   int64_t n_query, int32_t* out_idx, uint32_t* out_d2, float* out_dist,
                   uint8_t* out_pass, double ratio, sod_stream_t stream) {
  SOD_CHECK_ARG(n_parts >= 0 && n_query >= 0, "negative size");
  if (n_query == 0) return SOD_OK;
  SOD_CHECK_ARG(out_idx && out_d2, "null output pointer");
  SOD_CHECK_ARG(n_parts == 0 || (parts_idx && parts_d2), "null parts pointer");
  const int threads = 128;
  top2_merge_kernel<<<static_cast<unsigned>((n_query + threads - 1) / threads), threads, 0,
                      static_cast<cudaStream_t>(stream)>>>(parts_idx, parts_d2, n_parts, n_query,
                                                           out_idx, out_d2, out_dist, out_pass, ratio);
  SOD_CHECK_LAUNCH("top2_merge_kernel");
  return SOD_OK;
}

int sod_top2_keys(const int32_t* idx, const uint32_t* d2, int64_t n_query, int64_t n_rows, int64_t* keys,
                  sod_stream_t stream) {
  SOD_CHECK_ARG(n_query >= 0 && n_rows >= n_query, "need 0 <= n_query <= n_rows");
  if (n_rows == 0) return SOD_OK;
  SOD_CHECK_ARG(keys && (n_query == 0 || (idx && d2)), "null pointer");
  SOD_CHECK_ARG((reinterpret_cast<uintptr_t>(keys) & 15) == 0, "keys must be 16-byte aligned");
  const int threads = 256;
  top2_keys_kernel<<<static_cast<unsigned>((n_rows + threads - 1) / threads), threads, 0,
                     static_cast<cudaStream_t>(stream)>>>(idx, d2, n_query, n_rows,
                                                          reinterpret_cast<longlong2*>(keys));
  SOD_CHECK_LAUNCH("top2_keys_kernel");
  return SOD_OK;
}

int sod_top2_merge_keys(const int64_t* parts, int32_t n_parts, int64_t n_rows, int64_t* out, sod_stream_t stream) {
  SOD_CHECK_ARG(n_parts >= 0 && n_rows >= 0, "negative size");
  if (n_rows == 0) return SOD_OK;
  SOD_CHECK_ARG(out && (n_parts == 0 || parts), "null pointer");
  SOD_CHECK_ARG((reinterpret_cast<uintptr_t>(parts) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0,
                "key arrays must be 16-byte aligned");
  const int threads = 256;
  top2_merge_keys_kernel<<<static_cast<unsigned>((n_rows + threads - 1) / threads), threads, 0,
                           static_cast<cudaStream_t>(stream)>>>(reinterpret_cast<const longlong2*>(parts), n_parts,
                                                                n_rows, reinterpret_cast<longlong2*>(out));
  SOD_CHECK_LAUNCH("top2_merge_keys_kernel");
  return SOD_OK;
}

int sod_top2_from_keys(const int64_t* keys, int64_t n_query, int32_t* out_idx, uint32_t* out_d2, float* out_dist,
                       uint8_t* out_pass, double ratio, sod_stream_t stream) {
  SOD_CHECK_ARG(n_query >= 0, "negative size");
  if (n_query == 0) return SOD_OK;
  SOD_CHECK_ARG(keys && out_idx && out_d2, "null pointer");
  SOD_CHECK_ARG((reinterpret_cast<uintptr_t>(keys) & 15) == 0, "keys must be 16-byte aligned");
  const int threads = 256;
  top2_from_keys_kernel<<<static_cast<unsigned>((n_query + threads - 1) / threads), threads, 0,
                          static_cast<cudaStream_t>(stream)>>>(reinterpret_cast<const longlong2*>(keys), n_query,
                                                               out_idx, out_d2, out_dist, out_pass, ratio);
  SOD_CHECK_LAUNCH("top2_from_keys_kernel");
  return SOD_OK;
}

}  // extern "C"
