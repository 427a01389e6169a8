// ftsgemm_kernel.cuh -- the fused online-ABFT SGEMM kernel for sm_100a (B200).
//
// Replaces the reference's code-generated CUDA-core kernels
//   sgemm_{small..huge}    (/root/reference/kernel/ft_sgemm/include_code_gen/sgemm_*.cuh:11)     [FT = false]
//   ft_sgemm_{small..huge} (/root/reference/kernel/ft_sgemm/include_code_gen/ft_sgemm_*.cuh:11)  [FT = true]
// with ONE warp-specialised, persistent tcgen05 kernel template <BN, FT, CG>:
//
//   CG = 1 : one CTA per tile, UMMA 128 x BN x 8 (cta_group::1)
//   CG = 2 : a CTA PAIR (cluster of 2 on one TPC) per 256 x BN tile, UMMA 256 x BN x 8 (cta_group::2): each CTA stages
//            its own 128 rows of A and its own HALF of the B tile, so per-SM shared-memory traffic per flop halves --
//            the limiter measured on B200 (profiles/r01_ncu_*_v1.txt: TMA writes + UMMA reads share ~128 B/clk/SM)
//
//   warp 0   TMA producer   : cp.async.bulk.tensor 32(M|N) x 32(K) fp32 boxes, 128B swizzle with 32B atoms, into a
//                             STAGES-deep shared-memory ring (full/empty mbarriers)
//   warp 1   MMA issuer     : one thread (of the pair's leader CTA) issues tcgen05.mma.kind::tf32, FP32 accumulate in
//                             TMEM, two accumulator stages so the epilogue of tile i overlaps the main loop of tile i+1
//   warp 2   TMEM allocator
//   warps 4-7 epilogue      : tcgen05.ld (lane = row), per-row ABFT detect / locate / correct, C = alpha*acc + beta*C
//   warps 8-11 helpers      : (a) seeding tensor memory with the parked accumulator of the previous K-piece of a cut
//                             tile (plan.h), (b) the upper half of the columns of every final data-tile epilogue
//
// ABFT scheme (DESIGN.md section 3).  With b~ = the TF32 value the tensor core actually consumes and J_t the columns
// of N-tile t:
//   encode    (pre-pass encode_b_kernel; reference ENCODE ft_sgemm_huge.cuh:150-168)
//             e_t[k] = sum_{n in J_t} b~[n,k]      w_t[k] = sum_{n in J_t} (n-n0+1) b~[n,k]     (2-way TF32 split each)
//   checksum GEMM (reference CHECKSUM-GEMV :171-213): the 4 checksum vectors of every N-tile are appended to B as extra
//             "rows", i.e. the SAME kernel computes extra tile-columns  R = A * [e_t, w_t]^T  first (FP32 accumulate in
//             TMEM, identical operand rounding), writes them to a small workspace and publishes a per-32-row flag.
//             Cost: 4 columns per BN data columns (1.6 % at BN = 256) instead of a second pass over A.
//   detect    (epilogue; reference :328-421)  d1[m] = r1[m] - sum_n acc[m,n],  d2[m] = r2[m] - sum_n (n-n0+1) acc[m,n],
//             flagged iff |d1| > tau_abs + tau_rel * sum_n |acc[m,n]|
//   locate    column j = round(d2/d1) - 1   (weighted checksum; the reference intersects a row and a column residual)
//   correct   acc[m,j] = r1[m] - sum_{n != j} acc[m,n]   (recomputed, so Inf/NaN/huge upsets are repaired too;
//             reference :422-485 adds the row residual)
// One error per (row, tile) is correctable, i.e. up to 128 per CTA tile (the reference: one per tile per check).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <math_constants.h>

#include "ptx.cuh"

namespace ftsgemm {

constexpr int kBM = 128;          // rows per CTA (UMMA M = 128 * CG)
constexpr int kBK = 32;           // K extent of one shared-memory stage (4 UMMA k-steps of 8)
constexpr int kAtomMN = 32;       // floats per 128-byte swizzle row
constexpr int kChkPerTile = 4;    // checksum columns per N-tile: e hi/lo, w hi/lo (2 x 11-bit TF32 terms = 2^-22 relative)
constexpr int kThreads = 384;     // 12 warps: producer, MMA, TMEM alloc, idle, 4 epilogue, 4 helpers
constexpr int kMaxPeers = 16;     // ranks of one box whose verdict mailboxes a launch can write to
constexpr int kPeerSlotDoubles = 16;  // mailbox slot of one rank: 8 x (verdict double, sequence number), 16-byte pairs
constexpr int kMaxFaults = 8;
constexpr int kMaxEvents = 16;

struct DeviceFault {
  int row, col, mode;
  float add_value;
  unsigned int xor_mask;
};
struct DeviceEvent {
  int row, col;
  float residual, corrected_value;
  int status;
};
struct DeviceStats {
  unsigned long long tiles, rows_checked, detected, corrected, uncorrectable, checksum_faults;
  unsigned int max_abs_bits, max_rel_bits;
  int n_events;
  DeviceEvent events[kMaxEvents];
  unsigned long long recomputed;  // rows that were detected but not cleanly correctable and were recomputed on CUDA cores
  unsigned long long epilogue_faults;  // row segments whose store pass failed its check (protect_epilogue)
};

struct KernelParams {
  int M, N, K;
  float *C;
  int ldc;
  float alpha, beta;
  // tile schedule (tiles_m counts CG*128-row blocks)
  int tiles_m, tiles_n, group_n;
  // UMMA shared-memory descriptor parameters (runtime so the bring-up probe can sweep them)
  unsigned int lbo_bytes, sbo_bytes, layout_type, kstep_bytes;
  // bit 0 / 1 / 2: the A / B / checksum tensor map is 3-D {32, K, rows/32} so that ONE TMA instruction fetches a whole
  // operand stage (rows % 32 == 0); otherwise the map is 2-D {rows, K} and a stage takes one instruction per 32-row atom
  int tma3d;
  int dbg_flags;        // experiments only: bit 0 = skip the epilogue ABFT check of data tiles (timing breakdowns)
  // Work plan (built on the host, plan.h): unit u executes items plan[plan_off[u] .. plan_off[u+1]) in order.
  //   item.x = tile (decode order: checksum tiles first), item.y = kb_begin | kb_end << 16,
  //   item.z = kind (0 whole tile, 1 first piece, 3 middle piece, 2 last piece of a cut tile) | piece << 8,
  //   item.w = index among the cut tiles
  // The last sk_tiles data tiles are cut along K into up to sk_slices pieces so that the list scheduler can level the
  // units' finishing times.  Piece p parks its raw accumulator; piece p+1 loads it into tensor memory BEFORE its first
  // UMMA ("seed"), so a cut tile accumulates in exactly the k order of an uncut one (bit-identical).
  const int4 *plan;
  const int *plan_off;
  int sk_tiles, sk_slices;
  float *sk_ws;         // per (piece < sk_slices-1, cut tile, CTA of the group): one raw 128 x BN accumulator tile
  int *sk_flags;        // [((piece*sk_tiles + cut tile)*CG + cta_rank)*4 + quadrant] = sk_epoch once written
  int sk_epoch;
  // fault tolerance: checksum tile-columns
  int tiles_c;          // number of BN-wide checksum tile-columns (0 when FT is off)
  int chk_in_carriers;  // 1: no checksum tiles in the work plan -- the first data tile of every tile-row (plan kind 6, always the
                        // first item of its unit, when tensor-memory stage 1 is still free) also accumulates that row's
                        // checksum product R = A [e, w]^T in columns [BN, BN + n_chk_cols) and publishes it before its own
                        // check.  Costs ~0.25 tile-times per tile-row (the A slab is read from shared memory twice per
                        // k-step) instead of a 0.68 tile-time checksum item that streams A from HBM a second time.
  int chk_slices;       // >= 1: every checksum tile is computed as chk_slices independent K-slices (one plan item each, on
                        // otherwise idle units of small problems, where the checksum item is the critical path: its K loop
                        // starts after the encode and is as long as a data tile's); slice s publishes its partial expected
                        // checksums in plane s of chk_out / chk_flags, the check adds the planes in slice order
  int chk_box_bytes;    // bytes one CTA's TMA box of the checksum operand delivers per stage (<= kBBytes: the box is
                        // sized to the checksum columns that exist, so checksum items load less than data tiles)
  int n_chk_cols;       // tiles_n * kChkPerTile
  float *chk_out;       // M x n_chk_cols, column-major (ld = M): expected checksums r1/r2 (hi, lo each)
  int *chk_flags;       // [slab * tiles_c + c] = chk_epoch once checksum tile-column c of that 32-row slab is published
  int chk_epoch;
  // wave re-synchronisation (large problems): the leader producers form a barrier at every whole-tile boundary, so that
  // the units keep streaming the same k range of the A / B panels they share (without it the start times drift apart by
  // ~2 us per wave and the tile time grows 17 % over the 56 waves of 16384^3, profiles/r01_trace_*_16384*)
  int *wave_cnt;        // [w] = leader producers that have issued the last load of their w-th whole tile (cleared per launch)
  const int *wave_target;  // [w] = number of units that own more than w whole tiles
  int epi_assist;       // 1: the helper warp of each TMEM lane quadrant takes the upper half of the columns of every final
                        //    data-tile epilogue (check sums + store pass), halving the epilogue the units expose at the
                        //    end of their lists -- and the whole epilogue of a one-wave problem
  int pdl_wait;         // 1: launched as a programmatic dependent of the encode pre-pass -- checksum items (the only
                        //    consumers of its output) execute griddepcontrol.wait before their first load
                        // 2: launched as a programmatic dependent of whatever precedes it in the stream: every thread
                        //    executes griddepcontrol.wait after the prologue (barrier init, tensor-memory allocation), so
                        //    that only the launch latency and the prologue overlap the predecessor's tail
  // Small B (it fits L2 several times over): the encode runs as a FRONT PHASE of this kernel instead of a pre-pass launch --
  // all twelve warps of every CTA reduce their share of B (about one 8 KiB item per warp) before the roles start, then
  // add 1 to enc_done; the checksum items wait for enc_done to reach enc_target.  Saves the pre-pass's launch, drain and
  // the GEMM's exposed prologue (~3.5 us per step: 10 % at 2048^3); for large B the stand-alone pre-pass (16 warps per SM,
  // HBM-bound) is faster.
  int enc_front;
  float *enc_out;       // checksum operand [K][enc_ld]
  int enc_ld;
  int *enc_done;        // monotonic counter: warps that have finished their share, over all launches
  int enc_target;
  float tau_abs, tau_rel;
  int detect_only;
  // Fallback for rows that are flagged but cannot be repaired from the two checksums (upset too small to locate, two
  // upsets in one row, second checksum disagrees): the row segment of this tile is RECOMPUTED from A and B on CUDA cores
  // (TF32-truncated operands, FP32 accumulate) and written straight to C; the store pass skips it.  Nothing that was
  // detected is stored as computed.  (The reference only ever adds the residual, ft_sgemm_huge.cuh:422-485.)
  int recompute;
  const float *A, *B;   // the operands in global memory (lda = M, ldb = N)
  int lda, ldb;
  int inject_mode;
  float selftest_value;
  int selftest_row, selftest_col;
  int n_faults;
  DeviceFault faults[kMaxFaults];
  DeviceStats *stats;
  // Multi-GPU verdict exchange FUSED into this kernel (tile-sharded products, sharding.py): the last CTA of the grid to
  // finish writes this rank's verdict vector (the handle's counters, as ftsgemm_stats_device reports them) and the launch's
  // sequence number into slot peer_rank of EVERY rank's mailbox -- plain stores to peer memory over NVLink (the mailboxes
  // are mapped through CUDA IPC) -- so the exchange needs no collective kernel and nothing on the step's critical path but
  // ~2 us of one thread.  peer_world = 0: off.
  double *peer_box[kMaxPeers];
  int peer_world, peer_rank;
  double peer_seq;
  unsigned int *exit_count;  // CTAs of this launch that have finished (the last one resets it)
  // debug timeline (ftsgemm_debug_trace): per unit and item 8 x u64 = %globaltimer ns at {producer start, producer end,
  // MMA start, MMA issue end, epilogue start (accumulator complete), after check/fold, epilogue end}, tile | kind << 24
  unsigned long long *trace;
  int trace_cap;        // items recorded per unit
};

__device__ __forceinline__ unsigned long long globaltimer_ns() { return ptx::globaltimer(); }
__device__ __forceinline__ void trace_put(const KernelParams &p, int unit, int item, int slot, unsigned long long v) {
  if (p.trace != nullptr && item < p.trace_cap) p.trace[(static_cast<size_t>(unit) * p.trace_cap + item) * 8 + slot] = v;
}

#ifndef FTSGEMM_MAX_STAGES
#define FTSGEMM_MAX_STAGES 8
#endif

template <int BN, bool FT, int CG>
struct TileCfg {
  static_assert(CG == 1 || CG == 2, "cta_group");
  static_assert(BN % (32 * CG) == 0 && BN >= 32 && BN <= 256, "tile N");
  static constexpr int kBNLocal = BN / CG;                  // B rows staged by this CTA
  static constexpr int kABytes = kBM * kBK * 4;
  static constexpr int kBBytes = kBNLocal * kBK * 4;
  static constexpr int kOperandBytes = kABytes + kBBytes;
  // ABFT instantiations keep one 4 KiB slot per stage for a box of the checksum operand (one 32-column atom per CTA): a
  // CARRIER tile (plan item kind 6) loads it next to its own A / B stage and issues a second UMMA per k-step on the same A
  // slab, so the checksum product of its tile-row rides along instead of being a work item of its own.  The ring gets one
  // stage shorter for it (6 instead of 7 for the 256x256 pair tile: measured neutral, profiles/r02_ring_6_vs_7_stages.jsonl).
  // The slots form a ring of their own BEHIND the A / B stages (whose 32 KiB stride stays a power of two: with the slot
  // inside each stage -- a 36 KiB stride -- every main loop ran 21 % slower, profiles/r02_neg_stage_stride_36k.jsonl).
  static constexpr int kESlotBytes = FT ? kAtomMN * kBK * 4 : 0;
  static constexpr int kStageBytes = kOperandBytes;          // stride of the A / B ring
  static constexpr int kStageFootprint = kOperandBytes + kESlotBytes;
  static constexpr int kAccStages = (2 * BN <= 512) ? 2 : 1;
  static constexpr int kTmemNeeded = kAccStages * BN;
  static constexpr int kTmemCols = kTmemNeeded <= 32 ? 32 : kTmemNeeded <= 64 ? 64 : kTmemNeeded <= 128 ? 128
                                   : kTmemNeeded <= 256 ? 256 : 512;
  static constexpr int kBarBytes = 2048;  // barriers (512) + the epilogue pairs' exchange area (4 x 32 lanes x 3 floats)
  static constexpr int kMaxSmem = 227 * 1024 - 1024 /*alignment slack*/ - kBarBytes;
  static constexpr int kStagesFit = kMaxSmem / kStageFootprint;
  static constexpr int kStages = kStagesFit > FTSGEMM_MAX_STAGES ? FTSGEMM_MAX_STAGES : kStagesFit;
  static constexpr int kSmemBytes = kStages * kStageFootprint + 1024 + kBarBytes;
};

__device__ __forceinline__ float u2f(uint32_t u) { return __uint_as_float(u); }
__device__ __forceinline__ uint32_t f2u(float f) { return __float_as_uint(f); }

struct TileCoord {
  int m_blk, n_blk;  // n_blk indexes checksum tile-columns when is_chk
  int slice;         // K-slice of a checksum tile (0 otherwise)
  bool is_chk;
};

// Tile order: all checksum tile-columns first (so their results are published before the data tiles that need them
// reach their epilogue), then the data tiles in groups of group_n tile-columns, M fastest inside a group, so that one
// wave of CTAs shares few A row-panels and few B row-panels in L2.
__host__ __device__ __forceinline__ TileCoord decode_tile(const KernelParams &p, int t) {
  TileCoord tc;
  tc.slice = 0;
  const int per_slice = p.tiles_c * p.tiles_m;
  const int n_chk_tiles = p.chk_in_carriers ? 0 : per_slice * (p.chk_slices > 1 ? p.chk_slices : 1);
  if (t < n_chk_tiles) {
    tc.is_chk = true;
    tc.slice = t / (per_slice > 0 ? per_slice : 1);
    t -= tc.slice * per_slice;
    tc.m_blk = t % p.tiles_m;
    tc.n_blk = t / p.tiles_m;
    return tc;
  }
  t -= n_chk_tiles;
  tc.is_chk = false;
  const int per_group = p.group_n * p.tiles_m;
  const int g = t / per_group;
  const int first_n = g * p.group_n;
  const int gsz = p.group_n < p.tiles_n - first_n ? p.group_n : p.tiles_n - first_n;
  const int local = t - g * per_group;
  tc.n_blk = first_n + local % gsz;
  tc.m_blk = local / gsz;
  return tc;
}

// Checksum tile-column c covers checksum columns [c*BN, (c+1)*BN) (the last one fewer); its UMMA N is that width
// rounded up to 32*CG.  Measured: a checksum tile costs about as much as a data tile whatever its N, because its main
// loop is bound by the A-operand feed (L2 -> shared memory), not by the tensor pipe -- so checksum tile-columns are kept
// as wide as possible (narrow 64-column items made ABFT 5 % slower, profiles/r01_probe7_*), and only the last one is
// narrowed.
__host__ __device__ __forceinline__ int chk_cols_per_tile(int BN) { return BN; }
template <int BN, int CG>
__host__ __device__ __forceinline__ int chk_tile_width(const KernelParams &p, int c_blk) {
  const int cw = chk_cols_per_tile(BN);
  const int rest = p.n_chk_cols - c_blk * cw;
  const int cols = rest < cw ? rest : cw;
  const int q = 32 * CG;
  const int w = (cols + q - 1) / q * q;
  return w < BN ? w : BN;
}

// ------------------------------------------------------------------------------------------------------------
// Work decomposition.  Every role (producer, MMA issuer, epilogue) of work unit u walks the same item list, which the
// host built with a cost-aware list scheduler (plan.h).  Global item order = [checksum tiles][whole data tiles, raster
// order][split-K tail, slice-major]; each unit's list is increasing in that order and every wait (finisher ->
// contributors of the same tile, ABFT data tile -> checksum tiles) points to an EARLIER item, so the schedule cannot
// deadlock (tests/test_schedule.py simulates it, including the two-accumulator-stage constraint).  Slice-major order
// keeps all units on the same k-range of neighbouring tiles, so A/B panels stay shared in L2 (a contiguous stream-K
// split de-synchronised the k offsets and turned HBM-bound).
// ------------------------------------------------------------------------------------------------------------
struct Segment {
  int tile, kb_begin, kb_end;
  int kind;   // 0 whole tile, 1 first piece, 3 middle piece, 2 last piece, 6 carrier (whole data tile + its row's checksum product)
  int slice;
  int split_idx;
};

struct SegIter {
  const int4 *cur, *end;
  __device__ __forceinline__ SegIter(const KernelParams &p, int unit) {
    cur = p.plan + p.plan_off[unit];
    end = p.plan + p.plan_off[unit + 1];
  }
  __device__ __forceinline__ bool next(Segment &s) {
    if (cur == end) return false;
    const int4 e = __ldg(cur++);
    s.tile = e.x;
    s.kb_begin = e.y & 0xFFFF;
    s.kb_end = (e.y >> 16) & 0xFFFF;
    s.kind = e.z & 0xFF;
    s.slice = e.z >> 8;
    s.split_idx = e.w;
    return true;
  }
};

__device__ __forceinline__ int ld_acquire(const int *p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// ------------------------------------------------------------------------------------------------------------
// Epilogue store pass: out = alpha*acc + beta*out, column-major, lane = consecutive rows -> 128-byte coalesced.
// ------------------------------------------------------------------------------------------------------------
template <int BN>
__device__ __forceinline__ void store_tile(uint32_t taddr, float *crow, bool row_ok, int n0, int n_limit, int ldc,
                                           float alpha, float beta, int c_begin = 0, int c_end = BN / 32) {
  const bool full_n = (n0 + BN <= n_limit);
  if (full_n && beta != 0.0f) {
    // Software pipeline: the old values of chunk c + 1 are fetched while chunk c is stored (a chunk's 32 loads would
    // otherwise expose one L2 / HBM round trip per chunk, 4-8 in a row: the store pass is latency-, not bandwidth-bound).
    // (no per-lane control flow around the warp-collective tcgen05.ld: row_ok only predicates the global accesses)
    float old[32];
    if (row_ok) {
#pragma unroll
      for (int i = 0; i < 32; ++i) old[i] = crow[static_cast<size_t>(n0 + c_begin * 32 + i) * ldc];
    }
#pragma unroll 1
    for (int c = c_begin; c < c_end; ++c) {
      uint32_t v[32];
      __syncwarp();
      ptx::tmem_ld_x32(taddr + c * 32, v);
      ptx::tmem_wait_ld();
      const int nb = n0 + c * 32;
      if (row_ok) {
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = f2u(alpha * u2f(v[i]) + beta * old[i]);
        if (c + 1 < c_end) {
#pragma unroll
          for (int i = 0; i < 32; ++i) old[i] = crow[static_cast<size_t>(nb + 32 + i) * ldc];
        }
#pragma unroll
        for (int i = 0; i < 32; ++i) crow[static_cast<size_t>(nb + i) * ldc] = u2f(v[i]);
      }
    }
    return;
  }
#pragma unroll 1
  for (int c = c_begin; c < c_end; ++c) {
    uint32_t v[32];
    ptx::tmem_ld_x32(taddr + c * 32, v);
    ptx::tmem_wait_ld();
    const int nb = n0 + c * 32;
    if (!row_ok) continue;
    if (full_n) {
#pragma unroll
      for (int i = 0; i < 32; ++i) crow[static_cast<size_t>(nb + i) * ldc] = alpha * u2f(v[i]);
    } else {
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        if (nb + i < n_limit) {
          float *dst = crow + static_cast<size_t>(nb + i) * ldc;
          const float o = (beta == 0.0f) ? 0.0f : beta * (*dst);
          *dst = alpha * u2f(v[i]) + o;
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// ABFT check of one accumulator tile (executed by the 4 epilogue warps, lane = row).  Returns the column to replace
// (or -1) and its corrected value.  q = TMEM lane quadrant of this warp, m = global row of this lane.
// ------------------------------------------------------------------------------------------------------------
// The per-row sums of one chunk range of the accumulator (pass 1 of the check; also run by the assisting helper warp).
// Tensor-memory reads are the bound of this pass (64 B/clk per SM: 128 KiB of accumulator = ~1 us), so the next chunk's
// tcgen05.ld is in flight while this one is summed, and the sums run as two independent chains per quantity.
//   s2 = sum_j (j + 1) acc[j]  is formed per chunk as  (32 c + 1) * sum_i f_i + sum_i i * f_i   (i: compile-time weights)
__device__ __forceinline__ void abft_chunk_sums(const uint32_t (&v)[32], int c, float &s1, float &s2, float &sabs) {
  float a0 = 0.0f, a1 = 0.0f, t0 = 0.0f, t1 = 0.0f, b0 = 0.0f, b1 = 0.0f;
#pragma unroll
  for (int i = 0; i < 32; i += 2) {
    const float f0 = u2f(v[i]), f1 = u2f(v[i + 1]);
    a0 += f0;
    a1 += f1;
    t0 = fmaf(f0, static_cast<float>(i), t0);
    t1 = fmaf(f1, static_cast<float>(i + 1), t1);
    b0 += fabsf(f0);
    b1 += fabsf(f1);
  }
  const float sc = a0 + a1;
  s1 += sc;
  s2 += fmaf(static_cast<float>(c * 32 + 1), sc, t0 + t1);
  sabs += b0 + b1;
}
template <int BN>
__device__ __forceinline__ void abft_row_sums(uint32_t taddr, int c_begin, int c_end, float &s1, float &s2, float &sabs) {
  if (c_begin >= c_end) return;
  uint32_t va[32], vb[32];
  ptx::tmem_ld_x32(taddr + c_begin * 32, va);
  int c = c_begin;
#pragma unroll 1
  while (true) {
    ptx::tmem_wait_ld();
    ptx::tmem_ld_landed(va);
    const bool more_b = c + 1 < c_end;  // (warp-uniform)
    if (more_b) ptx::tmem_ld_x32(taddr + (c + 1) * 32, vb);
    abft_chunk_sums(va, c, s1, s2, sabs);
    if (!more_b) break;
    ptx::tmem_wait_ld();
    ptx::tmem_ld_landed(vb);
    const bool more_a = c + 2 < c_end;
    if (more_a) ptx::tmem_ld_x32(taddr + (c + 2) * 32, va);
    abft_chunk_sums(vb, c + 1, s1, s2, sabs);
    if (!more_a) break;
    c += 2;
  }
}

// c_mid < BN / 32: a helper warp of the same TMEM lane quadrant sums the chunks [c_mid, BN/32) and hands its three partial
// sums over through shared memory (xchg, 3 floats per lane) at named barrier pair_bar (64 threads); the same barrier
// also orders the injection before the helper's reads.
// The expected checksums of one row (4 floats published by the checksum tile-columns).  The epilogue warps try to fetch
// them BEFORE they wait for the accumulator (try_prefetch: the slab flag is polled once; when it is already raised the
// four loads are in flight during the wait), so that a flag round trip + a load round trip (~1.5 us) leave the critical
// path of every data-tile epilogue -- which is exposed at the end of every unit's list, and entirely in one-wave problems.
struct ExpectedChk {
  float e0, e1, w0, w1;
  bool ready;
};
__device__ __forceinline__ void load_expected(const KernelParams &p, int m, int n_blk, ExpectedChk &x) {
  x.e0 = x.e1 = x.w0 = x.w1 = 0.0f;
  if (m < p.M) {
    const float *cp = p.chk_out + static_cast<size_t>(n_blk) * kChkPerTile * p.M + m;
    x.e0 = __ldcg(cp);
    x.e1 = __ldcg(cp + p.M);
    x.w0 = __ldcg(cp + 2 * static_cast<size_t>(p.M));
    x.w1 = __ldcg(cp + 3 * static_cast<size_t>(p.M));
    const size_t plane = static_cast<size_t>(p.M) * p.n_chk_cols;
    for (int sl = 1; sl < p.chk_slices; ++sl) {  // K-slices of the checksum product, added in slice order (deterministic)
      cp += plane;
      x.e0 += __ldcg(cp);
      x.e1 += __ldcg(cp + p.M);
      x.w0 += __ldcg(cp + 2 * static_cast<size_t>(p.M));
      x.w1 += __ldcg(cp + 3 * static_cast<size_t>(p.M));
    }
  }
}
// number of flags per 32-row slab: checksum tile-columns x K-slices (flag index = slice * tiles_c + c)
__device__ __forceinline__ int chk_flags_per_slab(const KernelParams &p) { return p.tiles_c * (p.chk_slices > 1 ? p.chk_slices : 1); }
__device__ __forceinline__ void try_prefetch_expected(const KernelParams &p, int q, int lane, int m, int m0_cta, int n_blk,
                                                      ExpectedChk &x) {
  const int nf = chk_flags_per_slab(p);
  const int *flag = p.chk_flags + ((m0_cta >> 5) + q) * nf;
  int ok = 1;
  if (lane == 0)
    for (int c = 0; c < nf; ++c) ok &= (ld_acquire(flag + c) == p.chk_epoch) ? 1 : 0;
  ok = __shfl_sync(0xffffffffu, ok, 0);
  x.ready = ok != 0;
  if (x.ready) load_expected(p, m, n_blk, x);
}

template <int BN>
__device__ __forceinline__ void abft_check(const KernelParams &p, uint32_t taddr, int q, int lane, int m, int m0_cta,
                                           int n0, int n_blk, int &fix_col, float &fix_val, bool &redo, ExpectedChk &xp,
                                           float &own_s1, int c_mid = BN / 32, uint32_t xchg = 0u, int pair_bar = 0) {
  // ---- fault injection into the TMEM accumulator (reference: ft_sgemm_huge.cuh:324-327) ----
  if (p.inject_mode == 1) {
    if ((p.selftest_row >> 5) == q && p.selftest_col < BN) {
      uint32_t x = ptx::tmem_ld_x1(taddr + p.selftest_col);
      ptx::tmem_wait_ld();
      if (lane == (p.selftest_row & 31)) x = f2u(u2f(x) + p.selftest_value);
      ptx::tmem_st_x1(taddr + p.selftest_col, x);
      ptx::tmem_wait_st();
    }
  } else if (p.inject_mode == 2) {
    for (int f = 0; f < p.n_faults; ++f) {
      const int tr = p.faults[f].row - m0_cta, tc = p.faults[f].col - n0;
      if (p.faults[f].mode <= 1 && tr >= 0 && tr < kBM && tc >= 0 && tc < BN && (tr >> 5) == q) {  // warp-uniform
        uint32_t x = ptx::tmem_ld_x1(taddr + tc);
        ptx::tmem_wait_ld();
        if (lane == (tr & 31))
          x = p.faults[f].mode == 0 ? f2u(u2f(x) + p.faults[f].add_value) : (x ^ p.faults[f].xor_mask);
        ptx::tmem_st_x1(taddr + tc, x);
        ptx::tmem_wait_st();
      }
    }
  }
  const bool assisted = c_mid < BN / 32;
  if (assisted && p.inject_mode != 0) {  // the helper may only read the accumulator after the injection
    ptx::tc_fence_before();
    ptx::named_bar_sync(pair_bar, 64);
  }
  // ---- pass 1: actual row checksums (thread-local: lane == row) ----
  float s1 = 0.0f, s2 = 0.0f, sabs = 0.0f;
  abft_row_sums<BN>(taddr, 0, c_mid, s1, s2, sabs);
  own_s1 = s1;  // (this warp's columns only: what a protected store pass re-derives)
  if (assisted) {
    ptx::named_bar_sync(pair_bar, 64);  // the helper's partial sums are in shared memory
    s1 += ptx::ld_shared_f1(xchg + lane * 12);
    s2 += ptx::ld_shared_f1(xchg + lane * 12 + 4);
    sabs += ptx::ld_shared_f1(xchg + lane * 12 + 8);
  }
  // ---- expected checksums published by the checksum tile-columns (wait for this 32-row slab's flag unless the
  //      prefetch already found it raised) ----
  if (!xp.ready) {
    const int nf = chk_flags_per_slab(p);
    const int *flag = p.chk_flags + ((m0_cta >> 5) + q) * nf;
    if (lane == 0) {
      for (int c = 0; c < nf; ++c) {
        ptx::Watchdog wd;
        while (ld_acquire(flag + c) != p.chk_epoch) {
          __nanosleep(64);
          if (wd.tick()) break;
        }
      }
    }
    __syncwarp();
    load_expected(p, m, n_blk, xp);
  }
  const float r1 = xp.e0 + xp.e1, r2 = xp.w0 + xp.w1;
  const float d1 = r1 - s1, d2 = r2 - s2;
  const float thr = p.tau_abs + p.tau_rel * sabs;
  // Expected checksum AND row sum non-finite: Inf / NaN in the operands (this row of A, or a column of B in this tile), a
  // legitimately non-finite product that no checksum can verify.  Stored as computed, not flagged: recomputing it would only
  // re-round its finite elements (DESIGN.md section 3.3).  An upset makes one of the two non-finite, never both.
  const bool unverifiable = !isfinite(r1) && !isfinite(s1);
  const bool flagged = !unverifiable && !(fabsf(d1) <= thr);  // also true for NaN
  const unsigned flag_mask = __ballot_sync(0xffffffffu, flagged);

  // fault-free residual statistics (threshold calibration, DESIGN.md section 5)
  {
    float ra = (flagged || unverifiable) ? 0.0f : fabsf(d1);
    float rr = (flagged || unverifiable) ? 0.0f : fabsf(d1) / fmaxf(sabs, 1e-30f);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      ra = fmaxf(ra, __shfl_xor_sync(0xffffffffu, ra, o));
      rr = fmaxf(rr, __shfl_xor_sync(0xffffffffu, rr, o));
    }
    if (lane == 0 && p.stats) {
      atomicMax(&p.stats->max_abs_bits, f2u(ra));
      atomicMax(&p.stats->max_rel_bits, f2u(rr));
      atomicAdd(&p.stats->rows_checked, 32ull);
      if (q == 0) atomicAdd(&p.stats->tiles, 1ull);
    }
  }
  if (flag_mask == 0u) return;

  // ---- rare slow path (warp-uniform): locate, recompute, verify ----
  int j = -1;
  bool use_argmax = false;
  if (flagged) {
    if (isfinite(d1) && isfinite(d2) && d1 != 0.0f) {
      const float jf = d2 / d1;
      const float jr = rintf(jf);
      // The weighted residual d2 carries ~BN/2 times the noise of d1, so a column index is only trusted when the
      // upset is well above the detection threshold (measured, profiles/r01_fault_campaign_*: smaller upsets were
      // sometimes "corrected" one column off); below that the row is reported as detected-but-not-locatable and left
      // untouched (the upset is then < 1 % of max|C|).
      const bool locatable = fabsf(d1) >= 6.0f * thr;
      if (fabsf(jf) < 0.5f && locatable) j = -2;  // d2 ~ 0: the expected checksum itself was hit, data are intact
      else if (locatable && jr >= 1.0f && jr <= static_cast<float>(BN) && fabsf(jf - jr) <= 0.25f)
        j = static_cast<int>(jr) - 1;
      else j = -1;
    } else {
      use_argmax = true;  // Inf/NaN in the row: the culprit is the non-finite / largest element
    }
  }
  if (__ballot_sync(0xffffffffu, use_argmax) != 0u) {
    float best = -1.0f;
    int bj = 0;
#pragma unroll 1
    for (int c = 0; c < BN / 32; ++c) {
      uint32_t v[32];
      ptx::tmem_ld_x32(taddr + c * 32, v);
      ptx::tmem_wait_ld();
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const float a = fabsf(u2f(v[i]));
        if (!(a <= best)) {  // NaN wins
          best = (a == a) ? a : CUDART_INF_F;
          bj = c * 32 + i;
        }
      }
    }
    if (use_argmax) j = bj;
  }
  float x1 = 0.0f, x2 = 0.0f, xabs = 0.0f;  // row checksums without column j
#pragma unroll 1
  for (int c = 0; c < BN / 32; ++c) {
    uint32_t v[32];
    ptx::tmem_ld_x32(taddr + c * 32, v);
    ptx::tmem_wait_ld();
    const float wbase = static_cast<float>(c * 32 + 1);
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      const float f = (c * 32 + i == j) ? 0.0f : u2f(v[i]);
      x1 += f;
      x2 = fmaf(f, wbase + static_cast<float>(i), x2);
      xabs += fabsf(f);
    }
  }
  if (!flagged) return;
  int status;
  float vc = 0.0f;
  if (j == -2) {
    status = 4;
  } else if (j < 0) {
    status = 3;
  } else {
    vc = r1 - x1;
    const float wj = static_cast<float>(j + 1);
    const float e2 = (r2 - x2) - wj * vc;  // the second checksum must agree with a single error at column j
    const float tol = static_cast<float>(BN) * (p.tau_abs + p.tau_rel * (xabs + fabsf(vc)));
    status = (fabsf(e2) <= tol) ? 1 : 3;
  }
  if (status == 1 && p.detect_only) status = 2;
  if (status == 3 && p.recompute && !p.detect_only && m < p.M) status = 5;
  if (status == 1) {
    fix_col = j;
    fix_val = vc;
  }
  redo = status == 5;
  if (p.stats) {
    atomicAdd(&p.stats->detected, 1ull);
    if (status == 1) atomicAdd(&p.stats->corrected, 1ull);
    if (status == 3) atomicAdd(&p.stats->uncorrectable, 1ull);
    if (status == 4) atomicAdd(&p.stats->checksum_faults, 1ull);
    if (status == 5) atomicAdd(&p.stats->recomputed, 1ull);
    const int slot = atomicAdd(&p.stats->n_events, 1);
    if (slot < kMaxEvents) {
      DeviceEvent ev;
      ev.row = m;
      ev.col = j >= 0 ? n0 + j : -1;
      ev.residual = d1;
      ev.corrected_value = vc;
      ev.status = status;
      p.stats->events[slot] = ev;
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// Protected store pass (opts.protect_epilogue; the reference's epilogue, ft_sgemm_huge.cuh:573-690, is unprotected, and so
// is the window between its last accumulator check and the store).  The warp re-derives, from the accumulator values it
// re-reads, the row sum the ABFT check verified -- same association, so any difference in the bits is an upset of tensor
// memory or of the read path after the check -- and sums what it stores: sum(out) must equal alpha * sum(acc) + beta *
// sum(old) within the rounding of n_cols fused multiply-adds (2 * 128 * 2^-24 of the magnitudes).  Returns true in the
// lanes (= rows) whose segment failed.  bad_col / bad_mask: test injector (ftsgemm_fault.mode 3), -1 = none.
// ------------------------------------------------------------------------------------------------------------
struct StoreVerdict {
  float resid;
  bool bad;
};
template <int BN>
__device__ __forceinline__ StoreVerdict store_tile_protected(uint32_t taddr, float *crow, bool row_ok, int n0, int ldc, float alpha,
                                                          float beta, int c_begin, int c_end, float chk_s1, bool chk_s1_valid,
                                                          int bad_col, uint32_t bad_mask) {
  float s1 = 0.0f, s2 = 0.0f, sabs = 0.0f, so0 = 0.0f, so1 = 0.0f, sold0 = 0.0f, sold1 = 0.0f, aold0 = 0.0f, aold1 = 0.0f;
  const bool rmw = beta != 0.0f;
  float old[32];
  if (row_ok && rmw) {
#pragma unroll
    for (int i = 0; i < 32; ++i) old[i] = crow[static_cast<size_t>(n0 + c_begin * 32 + i) * ldc];
  }
#pragma unroll 1
  for (int c = c_begin; c < c_end; ++c) {
    uint32_t v[32];
    __syncwarp();
    ptx::tmem_ld_x32(taddr + c * 32, v);
    ptx::tmem_wait_ld();
    abft_chunk_sums(v, c, s1, s2, sabs);
    const int nb = n0 + c * 32;
    if (row_ok) {
      if (rmw) {
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          sold0 += old[i];
          sold1 += old[i + 1];
          aold0 += fabsf(old[i]);
          aold1 += fabsf(old[i + 1]);
        }
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = f2u(alpha * u2f(v[i]) + beta * old[i]);
        if (c + 1 < c_end) {
#pragma unroll
          for (int i = 0; i < 32; ++i) old[i] = crow[static_cast<size_t>(nb + 32 + i) * ldc];
        }
      } else {
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = f2u(alpha * u2f(v[i]));
      }
      if (bad_col >= c * 32 && bad_col < c * 32 + 32) {
#pragma unroll
        for (int i = 0; i < 32; ++i)
          if (c * 32 + i == bad_col) v[i] ^= bad_mask;
      }
#pragma unroll
      for (int i = 0; i < 32; i += 2) {
        so0 += u2f(v[i]);
        so1 += u2f(v[i + 1]);
      }
#pragma unroll
      for (int i = 0; i < 32; ++i) crow[static_cast<size_t>(nb + i) * ldc] = u2f(v[i]);
    }
  }
  const float ref = alpha * s1 + beta * (sold0 + sold1);
  const float tol = 1.6e-5f * (fabsf(alpha) * sabs + fabsf(beta) * (aold0 + aold1)) + 1e-30f;
  StoreVerdict out;
  out.resid = (so0 + so1) - ref;
  const bool reread_differs = chk_s1_valid && f2u(s1) != f2u(chk_s1);
  // (a non-finite reference -- Inf / NaN already in the old C -- cannot be verified and is not an upset)
  out.bad = row_ok && (reread_differs || (isfinite(ref) && !(fabsf(out.resid) <= tol)));
  return out;
}

// ------------------------------------------------------------------------------------------------------------
// Recompute fallback (rare): one warp recomputes row m of the tile's BN columns from global memory -- the values the
// tensor core would have produced up to FP32 accumulation order (TF32-truncated operands: every product is exact in
// FP32) -- and writes C = alpha * acc + beta * C directly.  K iterations of 1 broadcast + BN/32 coalesced loads.
// ------------------------------------------------------------------------------------------------------------
// (scalars by value: a reference to the __grid_constant__ parameter block would force a local copy of all of it)
template <int BN>
__device__ __noinline__ void recompute_row(const float *A, const float *B, float *C, int lda, int ldb, int ldc, int N, int K,
                                           float alpha, float beta, int m, int n0, int lane) {
  constexpr int J = BN / 32;
  float acc[J];
#pragma unroll
  for (int j = 0; j < J; ++j) acc[j] = 0.0f;
  const float *a = A + m;
  const float *b = B + n0 + lane;
#pragma unroll 2
  for (int k = 0; k < K; ++k) {
    const float av = u2f(f2u(__ldg(a + static_cast<size_t>(k) * lda)) & 0xFFFFE000u);
    const float *bk = b + static_cast<size_t>(k) * ldb;
#pragma unroll
    for (int j = 0; j < J; ++j) {
      const float bv = (n0 + lane + 32 * j < N) ? u2f(f2u(__ldg(bk + 32 * j)) & 0xFFFFE000u) : 0.0f;
      acc[j] = fmaf(av, bv, acc[j]);
    }
  }
#pragma unroll
  for (int j = 0; j < J; ++j) {
    const int n = n0 + lane + 32 * j;
    if (n < N) {
      float *dst = C + m + static_cast<size_t>(n) * ldc;
      const float o = (beta == 0.0f) ? 0.0f : beta * (*dst);
      *dst = alpha * acc[j] + o;
    }
  }
}

// The whole protected store pass of one warp, out of line and with scalars by value: an opt-in path must not cost the
// common epilogue registers (inlined it pushed the kernel into spills), and a reference to the __grid_constant__ parameter
// block would force a local copy of all of it.  Row segments that fail are counted and, with beta == 0, recomputed from A
// and B (with beta != 0 the old values of C are already overwritten: reported as uncorrectable).
template <int BN>
__device__ __noinline__ void protected_store_pass(uint32_t taddr, const float *A, const float *B, float *C, int lda, int ldb, int ldc,
                                                  int N, int K, float alpha, float beta, DeviceStats *stats, bool can_recompute,
                                                  int m, int row0, bool row_ok, int n0, int c_begin, int c_end, float chk_s1,
                                                  bool chk_s1_valid, int bad_col, uint32_t bad_mask, int lane) {
  const StoreVerdict sv = store_tile_protected<BN>(taddr, C + m, row_ok, n0, ldc, alpha, beta, c_begin, c_end, chk_s1, chk_s1_valid,
                                                   bad_col, bad_mask);
  unsigned mask = __ballot_sync(0xffffffffu, sv.bad);
  if (mask == 0u) return;
  const bool can_fix = beta == 0.0f && can_recompute;
  if (sv.bad && stats) {
    atomicAdd(&stats->epilogue_faults, 1ull);
    atomicAdd(can_fix ? &stats->recomputed : &stats->uncorrectable, 1ull);
    const int slot = atomicAdd(&stats->n_events, 1);
    if (slot < kMaxEvents) {
      DeviceEvent ev;
      ev.row = m;
      ev.col = -1;
      ev.residual = sv.resid;
      ev.corrected_value = 0.0f;
      ev.status = can_fix ? 6 : 7;
      stats->events[slot] = ev;
    }
  }
  if (!can_fix) return;
  while (mask != 0u) {
    const int r = __ffs(mask) - 1;
    mask &= mask - 1u;
    if (c_end - c_begin == BN / 32) {
      recompute_row<BN>(A, B, C, lda, ldb, ldc, N, K, alpha, beta, row0 + r, n0, lane);
    } else {
      if constexpr (BN >= 64) recompute_row<BN / 2>(A, B, C, lda, ldb, ldc, N, K, alpha, beta, row0 + r, n0 + c_begin * 32, lane);
    }
  }
}

// Test injectors for upsets AFTER the accumulator check (ftsgemm_fault.mode 2: into tensor memory before the store pass
// re-reads it; mode 3: into the value about to be stored -- returns the tile column for this lane, -1 if none).
template <int BN>
__device__ __forceinline__ void inject_after_check(const KernelParams &p, uint32_t taddr, int q, int lane, int m0_cta, int n0) {
  for (int f = 0; f < p.n_faults; ++f) {
    const int tr = p.faults[f].row - m0_cta, tc = p.faults[f].col - n0;
    if (p.faults[f].mode == 2 && tr >= 0 && tr < kBM && tc >= 0 && tc < BN && (tr >> 5) == q) {  // warp-uniform
      uint32_t x = ptx::tmem_ld_x1(taddr + tc);
      ptx::tmem_wait_ld();
      if (lane == (tr & 31)) x ^= p.faults[f].xor_mask;
      ptx::tmem_st_x1(taddr + tc, x);
      ptx::tmem_wait_st();
    }
  }
}
template <int BN>
__device__ __forceinline__ int stored_value_fault(const KernelParams &p, int q, int lane, int m0_cta, int n0, int c_begin, int c_end,
                                                  uint32_t &mask) {
  int col = -1;
  if (p.inject_mode == 2)
    for (int f = 0; f < p.n_faults; ++f) {
      const int tr = p.faults[f].row - m0_cta, tc = p.faults[f].col - n0;
      if (p.faults[f].mode == 3 && tr >= 0 && tr < kBM && (tr >> 5) == q && lane == (tr & 31) && tc >= c_begin * 32 && tc < c_end * 32) {
        col = tc;
        mask = p.faults[f].xor_mask;
      }
    }
  return col;
}

// ------------------------------------------------------------------------------------------------------------
// Cut tiles (plan.h).  Epilogue warps (lane = row) of a non-final piece park the raw accumulator slab; helper warps of
// the unit that owns the next piece load it back INTO tensor memory before that piece's first UMMA.
// ------------------------------------------------------------------------------------------------------------
template <int BN>
__device__ __forceinline__ void sk_dump_partial(const KernelParams &p, uint32_t taddr, float *ws, int *flag, int lane) {
#pragma unroll 1
  for (int c = 0; c < BN / 32; ++c) {
    uint32_t v[32];
    ptx::tmem_ld_x32(taddr + c * 32, v);
    ptx::tmem_wait_ld();
#pragma unroll
    for (int i = 0; i < 32; ++i) __stcg(ws + (c * 32 + i) * kBM, u2f(v[i]));
  }
  __threadfence();
  __syncwarp();
  if (lane == 0) atomicExch(flag, p.sk_epoch);
}

// seed: the previous piece's parked accumulator goes back into tensor memory before this piece's first UMMA
template <int BN>
__device__ __forceinline__ void sk_seed(const KernelParams &p, uint32_t taddr, const float *ws, const int *flag, int lane) {
  if (lane == 0) {
    ptx::Watchdog wd;
    while (ld_acquire(flag) != p.sk_epoch) {
      __nanosleep(64);
      if (wd.tick()) break;
    }
  }
  __syncwarp();
#pragma unroll 1
  for (int c = 0; c < BN / 32; ++c) {
    uint32_t v[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = f2u(__ldcg(ws + (c * 32 + i) * kBM));
    ptx::tmem_st_x32(taddr + c * 32, v);
  }
  ptx::tmem_wait_st();
}

// ------------------------------------------------------------------------------------------------------------
// ENCODE of B (reference: ft_sgemm_huge.cuh:150-168, done there per CTA and per k-step with shuffles; here once per
// GEMM and per BN-wide column block -- a CUDA-core re-read of every shared-memory stage does not fit next to a
// tensor-core main loop, DESIGN.md section 3).
//   chk[k][t*4 + 0..1] = (hi, lo) TF32 split of  e = sum_{n in block t} tf32(B[n,k])
//   chk[k][t*4 + 2..3] = (hi, lo) TF32 split of  w = sum_{n in block t} (n - n0 + 1) * tf32(B[n,k])
// Each lane sums its <= 8 elements of a row in plain FP32 -- TF32 inputs have 11-bit significands and (j+1)*b is an
// exact 20-bit product, so these short sums are exact unless the elements differ by > 2^10 in magnitude -- the 32-way
// cross-lane reduction runs in FP64 as a transposing butterfly (NV values per lane -> one per lane: NV-1 + log steps
// instead of 5*NV shuffles), and the two TF32 terms carry each checksum to ~2^-22 relative.
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float tf32_bits(float x, int rounding) {
  uint32_t u = __float_as_uint(x);
  if (rounding == 1) u += 0x1000u;  // round-to-nearest (ties away), like cvt.rna.tf32.f32
  if (rounding != 2) u &= 0xFFFFE000u;
  return __uint_as_float(u);
}
__device__ __forceinline__ void split2_tf32(double x, float &h, float &l) {
  h = tf32_bits(static_cast<float>(x), 0);
  l = tf32_bits(static_cast<float>(x - static_cast<double>(h)), 0);  // x - h is exact in FP64
}

// v[0..CNT) per lane -> after all steps v[0] of lane L is the 32-lane total of value idx(L)
template <typename T, int CNT, int O>
struct TransposeReduce {
  static __device__ __forceinline__ void run(T *v, int lane, int &idx) {
    if constexpr (O > 0) {
      if constexpr (CNT > 1) {
        constexpr int H = CNT / 2;
        const bool up = (lane & O) != 0;
#pragma unroll
        for (int i = 0; i < H; ++i) {
          const T send = up ? v[i] : v[i + H];
          const T keep = up ? v[i + H] : v[i];
          v[i] = keep + __shfl_xor_sync(0xffffffffu, send, O);
        }
        if (up) idx += H;
        TransposeReduce<T, H, O / 2>::run(v, lane, idx);
      } else {
        v[0] += __shfl_xor_sync(0xffffffffu, v[0], O);
        TransposeReduce<T, 1, O / 2>::run(v, lane, idx);
      }
    }
  }
};

// One warp encodes items (column block t, KR consecutive k-rows), item = gw, gw + nw, ...; t fastest, so that warps
// running side by side read neighbouring 1 KiB segments of the same rows of B.
// 16-byte read-only load; STREAM: evict-first in L2 (B larger than L2: the pre-pass must not push the GEMM's working set
// -- the tails of A, B, C the previous launch left there -- out of the cache for data it will not find again anyway)
template <bool STREAM>
__device__ __forceinline__ float4 ld_b16(const float4 *p) {
  if (!STREAM) return __ldg(p);
  uint64_t policy;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p), "l"(policy));
  return v;
}

template <int BN, int KRQ, bool STREAM = false>
__device__ __forceinline__ void encode_b_warp(const float *__restrict__ B, int N, int K, int ldb, float *__restrict__ chk,
                                              int chk_ld, int rounding, int tiles_n, int gw, int nw, int lane) {
  constexpr int J = BN >= 128 ? BN / 128 : 0;   // float4 loads per lane and k-row
  constexpr int KR = (J == 2) ? KRQ : 2 * KRQ;  // k-rows per item: 2 * KRQ float4 (J = 2, 1) in flight per lane
  constexpr int NV = 2 * KR;
  if (J > 0 && N == tiles_n * BN && ldb == N) {
    // Linear path (every column block full, rows contiguous): B is one flat array of (k, t) segments of BN floats, k-major;
    // an item is KR CONSECUTIVE segments = one contiguous KR * BN * 4-byte read per warp (8 KiB), and its results are
    // KR consecutive float4 of the checksum operand.  (The strided item shape below -- KR k-rows of one column block --
    // fell from 5.6 TB/s at N = 4096 to 3.9 TB/s at N = 8192, where the rows are 32 KiB apart.)
    const long long pairs = static_cast<long long>(K) * tiles_n;
    const long long items = (pairs + KR - 1) / KR;
    for (long long item = gw; item < items; item += nw) {
      const long long q0 = item * KR;
      float4 x[KR][J > 0 ? J : 1];
#pragma unroll
      for (int u = 0; u < KR; ++u)
#pragma unroll
        for (int jj = 0; jj < J; ++jj)
          x[u][jj] = (q0 + u < pairs)
                         ? ld_b16<STREAM>(reinterpret_cast<const float4 *>(B + static_cast<size_t>(q0 + u) * BN) + lane + 32 * jj)
                         : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      double v[NV];
#pragma unroll
      for (int u = 0; u < KR; ++u) {
        float e = 0.0f, w = 0.0f;
#pragma unroll
        for (int jj = 0; jj < J; ++jj) {
          const float wj = static_cast<float>(4 * (lane + 32 * jj) + 1);
          const float b0 = tf32_bits(x[u][jj].x, rounding), b1 = tf32_bits(x[u][jj].y, rounding),
                      b2 = tf32_bits(x[u][jj].z, rounding), b3 = tf32_bits(x[u][jj].w, rounding);
          e += (b0 + b1) + (b2 + b3);
          w += (b0 * wj + b1 * (wj + 1.0f)) + (b2 * (wj + 2.0f) + b3 * (wj + 3.0f));
        }
        v[2 * u] = static_cast<double>(e);
        v[2 * u + 1] = static_cast<double>(w);
      }
      int idx = 0;
      TransposeReduce<double, NV, 16>::run(v, lane, idx);
      const long long q = q0 + (idx >> 1);
      if ((lane & (32 / NV - 1)) == 0 && q < pairs) {
        float h, l;
        split2_tf32(v[0], h, l);
        const int k = static_cast<int>(q / tiles_n), t = static_cast<int>(q - static_cast<long long>(k) * tiles_n);
        *reinterpret_cast<float2 *>(chk + static_cast<size_t>(k) * chk_ld + t * kChkPerTile + (idx & 1) * 2) = make_float2(h, l);
      }
    }
    return;
  }
  const int k_items = (K + KR - 1) / KR;
  const int total = tiles_n * k_items;
  for (int item = gw; item < total; item += nw) {
    const int t = item % tiles_n;
    const int n0 = t * BN;
    const int k0 = (item / tiles_n) * KR;
    double v[NV];
    if (J > 0 && n0 + BN <= N && k0 + KR <= K) {  // full block: 16-byte loads (ldb % 4 == 0, n0 % 4 == 0)
      float4 x[KR][J > 0 ? J : 1];
#pragma unroll
      for (int u = 0; u < KR; ++u)
#pragma unroll
        for (int jj = 0; jj < J; ++jj)
          x[u][jj] = ld_b16<STREAM>(reinterpret_cast<const float4 *>(B + static_cast<size_t>(k0 + u) * ldb + n0) + lane + 32 * jj);
#pragma unroll
      for (int u = 0; u < KR; ++u) {
        float e = 0.0f, w = 0.0f;
#pragma unroll
        for (int jj = 0; jj < J; ++jj) {
          const float wj = static_cast<float>(4 * (lane + 32 * jj) + 1);
          const float b0 = tf32_bits(x[u][jj].x, rounding), b1 = tf32_bits(x[u][jj].y, rounding),
                      b2 = tf32_bits(x[u][jj].z, rounding), b3 = tf32_bits(x[u][jj].w, rounding);
          e += (b0 + b1) + (b2 + b3);
          w += (b0 * wj + b1 * (wj + 1.0f)) + (b2 * (wj + 2.0f) + b3 * (wj + 3.0f));
        }
        v[2 * u] = static_cast<double>(e);
        v[2 * u + 1] = static_cast<double>(w);
      }
    } else {
#pragma unroll
      for (int u = 0; u < KR; ++u) {
        float e = 0.0f, w = 0.0f;
        const int k = k0 + u;
        if (k < K) {
          for (int j = lane; j < BN; j += 32) {
            if (n0 + j < N) {
              const float b = tf32_bits(__ldg(B + static_cast<size_t>(k) * ldb + n0 + j), rounding);
              e += b;
              w += b * static_cast<float>(j + 1);
            }
          }
        }
        v[2 * u] = static_cast<double>(e);
        v[2 * u + 1] = static_cast<double>(w);
      }
    }
    int idx = 0;
    TransposeReduce<double, NV, 16>::run(v, lane, idx);
    const int k = k0 + (idx >> 1);
    if ((lane & (32 / NV - 1)) == 0 && k < K) {
      float h, l;
      split2_tf32(v[0], h, l);
      *reinterpret_cast<float2 *>(chk + static_cast<size_t>(k) * chk_ld + t * kChkPerTile + (idx & 1) * 2) = make_float2(h, l);
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// The kernel.
// ------------------------------------------------------------------------------------------------------------
// PROT: the instantiation with the protected store pass (opts.protect_epilogue) -- a separate binary, because the common
// kernel sits exactly at the 168-register limit of a 384-thread CTA and every extra live value of an opt-in path spilled.
template <int BN, bool FT, int CG, bool PROT = false>
__global__ void __launch_bounds__(kThreads, 1)
ftsgemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                  const __grid_constant__ CUtensorMap tmChk, const KernelParams p) {
  using Cfg = TileCfg<BN, FT, CG>;
  constexpr int kStages = Cfg::kStages;
  constexpr int kAccStages = Cfg::kAccStages;

  extern __shared__ uint8_t smem_raw[];
  // 128B-swizzle atoms need 1024B alignment.  (Both CTAs of a pair see the same dynamic-smem base offset, which
  // cta_group::2 requires: the pair's MMA applies one descriptor to both CTAs' shared memory.)
  const uint32_t smem_base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t eslot_base = smem_base + kStages * Cfg::kStageBytes;  // checksum-operand slots of the carrier tiles
  const uint32_t bar_base = smem_base + kStages * Cfg::kStageFootprint;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kStages + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * kStages + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * kStages + 2 + a); };
  auto seeded_bar = [&](int a) { return bar_base + 8u * (2 * kStages + 4 + a); };  // leader: TMEM stage a holds the seed
  // carrier tiles: the epilogue warps (of both CTAs) have read the checksum columns out of tensor-memory stage 1
  const uint32_t chk_drained_bar = bar_base + 8u * (2 * kStages + 6);
  const uint32_t tmem_slot = bar_base + 8u * (2 * kStages + 7);
  // number of (epilogue warp, item) pairs this CTA has finished: the helper warps' view of which accumulator stages
  // are drained (a counter, not an mbarrier: the helpers may be many items behind while they encode B)
  const uint32_t epi_count = tmem_slot + 8u;
  auto xchg_base = [&](int q) { return bar_base + 512u + static_cast<uint32_t>(q) * (32u * 12u); };
  constexpr int kMid = BN / 64;  // chunks [0, kMid) to the epilogue warp, [kMid, BN/32) to its helper (BN >= 64)
  volatile uint32_t *tmem_slot_ptr =
      reinterpret_cast<volatile uint32_t *>(smem_raw + (tmem_slot - ptx::smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t cta_rank = (CG == 2) ? ptx::cluster_ctarank() : 0u;
  const bool is_leader = cta_rank == 0;
  const int unit = blockIdx.x / CG;        // persistent work unit = CTA (CG=1) or CTA pair (CG=2)

  // the next kernel in the stream (if it was launched as a programmatic dependent) may be scheduled as soon as this
  // grid's CTAs retire; it synchronises with griddepcontrol.wait itself
  ptx::pdl_launch_dependents();
  if (warp == 0 && lane == 0) {
    ptx::tma_prefetch_desc(&tmA);
    ptx::tma_prefetch_desc(&tmB);
    if (FT) ptx::tma_prefetch_desc(&tmChk);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < kStages; ++s) {
      ptx::mbar_init(full_bar(s), CG);   // leader's own arrive.expect_tx (+ the peer's remote arrive)
      ptx::mbar_init(empty_bar(s), 1);   // one tcgen05.commit (multicast to both CTAs when CG = 2)
    }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(tfull_bar(a), 1);
      ptx::mbar_init(tempty_bar(a), 4 * CG);  // one arrive per epilogue warp of every CTA in the group
      ptx::mbar_init(seeded_bar(a), 4 * CG);  // one arrive per helper warp of every CTA in the group
    }
    ptx::st_shared_u32(epi_count, 0u);
    ptx::mbar_init(chk_drained_bar, 4 * CG);
    ptx::fence_mbar_init();
  }
  if (CG == 2) ptx::cluster_sync_all();  // peer barriers must be initialised before any remote arrive / 2-CTA alloc
  if (warp == 2) {
    if (CG == 2) {
      ptx::tmem_alloc_cg2(tmem_slot, Cfg::kTmemCols);
      ptx::tmem_relinquish_cg2();
    } else {
      ptx::tmem_alloc(tmem_slot, Cfg::kTmemCols);
      ptx::tmem_relinquish();
    }
  }
  ptx::tc_fence_before();
  if (CG == 2) ptx::cluster_sync_all();
  else __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  if (p.pdl_wait == 2) ptx::pdl_wait();  // everything before this line touched no global memory

  if (FT && p.enc_front) {
    // front-phase ENCODE of B (see KernelParams::enc_front): the same routine as the pre-pass kernel
    const int gw = static_cast<int>(blockIdx.x) * (kThreads / 32) + warp, nw = static_cast<int>(gridDim.x) * (kThreads / 32);
    encode_b_warp<BN, 8>(p.B, p.N, p.K, p.ldb, p.enc_out, p.enc_ld, 0, p.tiles_n, gw, nw, lane);
    __syncwarp();  // the warp's stores are ordered before lane 0's release (cumulativity)
    if (lane == 0) {
      ptx::fence_acq_rel_gpu();
      atomicAdd(p.enc_done, 1);
    }
  }

  if (warp == 0) {
    // ===================================================================== TMA producer (every CTA)
    // warp-uniform loop, one elected lane issues the TMA instructions (see ptx::elect_one)
    int stage = 0;
    uint32_t phase = 0;
    SegIter it(p, unit);
    Segment sg;
    int item_idx = -1;
    bool pdl_done = false;
    int whole_ord = 0;  // whole data tiles this unit has loaded (wave index)
    while (it.next(sg)) {
      ++item_idx;
      const TileCoord tc = decode_tile(p, sg.tile);
      const int m0 = (tc.m_blk * CG + static_cast<int>(cta_rank)) * kBM;        // this CTA's 128 rows of A
      const bool b_is_chk = FT && tc.is_chk;
      const bool carrier = FT && sg.kind == 6;
      const bool wave_item = p.wave_cnt != nullptr && sg.kind == 0 && !b_is_chk && is_leader;
      if (wave_item && whole_ord > 0) {
        // all units have finished loading their previous whole tile: start this one together
        if (lane == 0) {
          ptx::Watchdog wd;
          const int need = __ldg(p.wave_target + whole_ord - 1);
          while (ld_acquire(p.wave_cnt + whole_ord - 1) < need) {
            __nanosleep(32);
            if (wd.tick()) break;
          }
        }
        __syncwarp();
      }
      const int n_eff = b_is_chk ? chk_tile_width<BN, CG>(p, tc.n_blk) : BN;
      const int nb0 = (b_is_chk ? tc.n_blk * chk_cols_per_tile(BN) : tc.n_blk * BN) +
                      static_cast<int>(cta_rank) * (n_eff / CG);  // this CTA's share of B rows
      const CUtensorMap *tmb = b_is_chk ? &tmChk : &tmB;
      if (FT && (b_is_chk || carrier) && p.pdl_wait == 1 && !pdl_done) {
        ptx::pdl_wait();  // the pre-pass kernel has completed and its writes are visible
        pdl_done = true;
      }
      if (FT && (b_is_chk || carrier) && p.enc_front && !pdl_done) {
        // front-phase encode: every warp of the grid has stored its share of the checksum operand
        if (lane == 0) {
          ptx::Watchdog wd;
          while (ld_acquire(p.enc_done) - p.enc_target < 0) {
            __nanosleep(64);
            if (wd.tick()) break;
          }
        }
        __syncwarp();
        ptx::fence_proxy_async();  // generic-proxy writes (st.global) -> async-proxy reads (TMA)
        pdl_done = true;
      }
      if (p.trace != nullptr && is_leader && lane == 0) trace_put(p, unit, item_idx, 0, globaltimer_ns());
      // The loop body is specialised OUTSIDE the k loop: with 3-D tensor maps a stage is exactly two TMA instructions
      // (predicated-off TMA instructions still cost issue time on the single producer thread).
      const bool all3d = (p.tma3d & 1) && (p.tma3d & (b_is_chk ? 4 : 2));
      const int a_atom = m0 / kAtomMN, b_atom = nb0 / kAtomMN;
      // (the B descriptor is a kernel-parameter address known at compile time in each copy of the loop: a run-time
      //  selected descriptor pointer measurably slows the TMA issue)
      auto fast_loop = [&](const CUtensorMap *tmb_const) {
        const uint32_t stage_tx = b_is_chk ? static_cast<uint32_t>(Cfg::kABytes + p.chk_box_bytes)
                                           : static_cast<uint32_t>(Cfg::kOperandBytes);
        for (int kb = sg.kb_begin; kb < sg.kb_end; ++kb) {
          ptx::mbar_wait(empty_bar(stage), phase ^ 1u);
          const uint32_t sA = smem_base + stage * Cfg::kStageBytes;
          const uint32_t sB = sA + Cfg::kABytes;
          const int k0 = kb * kBK;
          if (ptx::elect_one()) {
            if (CG == 2) {
              const uint32_t bar = ptx::mapa(full_bar(stage), 0);  // the leader's barrier collects both CTAs' bytes
              if (is_leader) ptx::mbar_arrive_expect_tx(full_bar(stage), 2 * stage_tx);
              else ptx::mbar_arrive_cluster(bar);
              ptx::tma_load_3d_cg2(sA, &tmA, bar, 0, k0, a_atom);
              ptx::tma_load_3d_cg2(sB, tmb_const, bar, 0, k0, b_atom);
            } else {
              ptx::mbar_arrive_expect_tx(full_bar(stage), stage_tx);
              ptx::tma_load_3d(sA, &tmA, full_bar(stage), 0, k0, a_atom);
              ptx::tma_load_3d(sB, tmb_const, full_bar(stage), 0, k0, b_atom);
            }
          }
          __syncwarp();
          if (++stage == kStages) {
            stage = 0;
            phase ^= 1u;
          }
        }
      };
      // carrier tile: the same loop with a third load per stage (the loops are specialised OUTSIDE the k loop: a predicated-off
      // TMA / UMMA instruction in the ordinary loops cost every tile 20 % -- the issue threads are the bottleneck)
      auto carrier_loop = [&]() {
        const uint32_t stage_tx = static_cast<uint32_t>(Cfg::kOperandBytes + p.chk_box_bytes);
        const int e_atom = static_cast<int>(cta_rank) * (p.chk_box_bytes / (kAtomMN * kBK * 4));  // this CTA's share of [e, w]
        for (int kb = sg.kb_begin; kb < sg.kb_end; ++kb) {
          ptx::mbar_wait(empty_bar(stage), phase ^ 1u);
          const uint32_t sA = smem_base + stage * Cfg::kStageBytes;
          const uint32_t sB = sA + Cfg::kABytes;
          const uint32_t sE = eslot_base + stage * Cfg::kESlotBytes;
          const int k0 = kb * kBK;
          if (ptx::elect_one()) {
            if (CG == 2) {
              const uint32_t bar = ptx::mapa(full_bar(stage), 0);
              if (is_leader) ptx::mbar_arrive_expect_tx(full_bar(stage), 2 * stage_tx);
              else ptx::mbar_arrive_cluster(bar);
              ptx::tma_load_3d_cg2(sA, &tmA, bar, 0, k0, a_atom);
              ptx::tma_load_3d_cg2(sB, &tmB, bar, 0, k0, b_atom);
              ptx::tma_load_3d_cg2(sE, &tmChk, bar, 0, k0, e_atom);
            } else {
              ptx::mbar_arrive_expect_tx(full_bar(stage), stage_tx);
              ptx::tma_load_3d(sA, &tmA, full_bar(stage), 0, k0, a_atom);
              ptx::tma_load_3d(sB, &tmB, full_bar(stage), 0, k0, b_atom);
              ptx::tma_load_3d(sE, &tmChk, full_bar(stage), 0, k0, e_atom);
            }
          }
          __syncwarp();
          if (++stage == kStages) {
            stage = 0;
            phase ^= 1u;
          }
        }
      };
      if (FT && carrier) {
        carrier_loop();
      } else if (all3d) {
        if (b_is_chk) fast_loop(&tmChk);
        else fast_loop(&tmB);
      } else {
        for (int kb = sg.kb_begin; kb < sg.kb_end; ++kb) {
          ptx::mbar_wait(empty_bar(stage), phase ^ 1u);
          const uint32_t sA = smem_base + stage * Cfg::kStageBytes;
          const uint32_t sB = sA + Cfg::kABytes;
          const int k0 = kb * kBK;
          const uint32_t bar = (CG == 2) ? ptx::mapa(full_bar(stage), 0) : full_bar(stage);
          const uint32_t stage_tx = (b_is_chk && (p.tma3d & 4)) ? static_cast<uint32_t>(Cfg::kABytes + p.chk_box_bytes)
                                                                : static_cast<uint32_t>(Cfg::kOperandBytes);
          if (ptx::elect_one()) {
          if (CG == 2) {
            if (is_leader) ptx::mbar_arrive_expect_tx(full_bar(stage), 2 * stage_tx);
            else ptx::mbar_arrive_cluster(bar);
          } else {
            ptx::mbar_arrive_expect_tx(full_bar(stage), stage_tx);
          }
          if (p.tma3d & 1) {
            if (CG == 2) ptx::tma_load_3d_cg2(sA, &tmA, bar, 0, k0, a_atom);
            else ptx::tma_load_3d(sA, &tmA, bar, 0, k0, a_atom);
          } else {
#pragma unroll
            for (int i = 0; i < kBM / kAtomMN; ++i) {
              if (CG == 2) ptx::tma_load_2d_cg2(sA + i * (kBK * 128), &tmA, bar, m0 + i * kAtomMN, k0);
              else ptx::tma_load_2d(sA + i * (kBK * 128), &tmA, bar, m0 + i * kAtomMN, k0);
            }
          }
          if (p.tma3d & (b_is_chk ? 4 : 2)) {
            if (CG == 2) ptx::tma_load_3d_cg2(sB, tmb, bar, 0, k0, b_atom);
            else ptx::tma_load_3d(sB, tmb, bar, 0, k0, b_atom);
          } else {
#pragma unroll
            for (int i = 0; i < Cfg::kBNLocal / kAtomMN; ++i) {
              if (CG == 2) ptx::tma_load_2d_cg2(sB + i * (kBK * 128), tmb, bar, nb0 + i * kAtomMN, k0);
              else ptx::tma_load_2d(sB + i * (kBK * 128), tmb, bar, nb0 + i * kAtomMN, k0);
            }
          }
          }
          __syncwarp();
          if (++stage == kStages) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
      if (wave_item) {
        if (lane == 0) atomicAdd(p.wave_cnt + whole_ord, 1);
        ++whole_ord;
      }
      if (p.trace != nullptr && is_leader && lane == 0) trace_put(p, unit, item_idx, 1, globaltimer_ns());
    }
  } else if (warp == 1 && is_leader) {
    // ===================================================================== MMA issuer (leader CTA only)
    // The whole warp walks the loop (uniform control flow); one elected lane issues the UMMAs and their commits.
    const uint32_t idesc = ptx::make_idesc_tf32(kBM * CG, BN, 1, 1);
    const uint64_t desc0 = ptx::make_smem_desc(smem_base, p.lbo_bytes, p.sbo_bytes, p.layout_type);
    const uint64_t desc_hi = desc0 & 0xFFFFFFFF00000000ull;
    const uint32_t desc_lo0 = static_cast<uint32_t>(desc0);
    const uint32_t kstep16 = p.kstep_bytes >> 4;
    const uint32_t e_lo0 = desc_lo0 + ((eslot_base - smem_base) >> 4);  // checksum-operand slot of stage 0 (carrier tiles)
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    uint32_t seed_phase = 0;  // bit a: parity of seeded_bar(a)
    bool first_is_carrier = false;
    SegIter it(p, unit);
    Segment sg;
    int item_idx = -1;
    while (it.next(sg)) {
      ++item_idx;
      uint32_t idesc_t = idesc;
      const bool carrier = FT && sg.kind == 6;
      uint32_t idesc_c = 0u;
      if (FT) {
        const TileCoord tc = decode_tile(p, sg.tile);
        if (tc.is_chk) idesc_t = ptx::make_idesc_tf32(kBM * CG, chk_tile_width<BN, CG>(p, tc.n_blk), 1, 1);
        if (carrier) idesc_c = ptx::make_idesc_tf32(kBM * CG, chk_tile_width<BN, CG>(p, 0), 1, 1);
        // a carrier is the first item of its unit and also occupies accumulator stage 1: the second item may only start
        // once the carrier's epilogue has read the checksum columns out of it
        if (item_idx == 1 && first_is_carrier) {
          ptx::mbar_wait(chk_drained_bar, 0u);
          ptx::tc_fence_after();
        }
        if (item_idx == 0) first_is_carrier = carrier;
      }
      ptx::mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
      ptx::tc_fence_after();
      if (p.trace != nullptr && lane == 0) trace_put(p, unit, item_idx, 2, globaltimer_ns());
      const uint32_t d_tmem = tmem_base + acc * BN;
      // Lean issue loop: a single thread runs dependent integer chains at ~1 instruction per 4-6 cycles, and four UMMAs
      // (one k-block) take only ~512 cycles, so the 64-bit descriptors are NOT rebuilt per UMMA: the high word
      // (SBO, version, layout) and LBO are constant, only the 14-bit start-address field advances (+64 = 1024 B).
      uint32_t first = 1u;  // the first UMMA of a tile overwrites the accumulator ...
      if (sg.kind == 2 || sg.kind == 3) {   // ... unless the helper warps seeded it with the previous piece's parked sums
        ptx::mbar_wait(seeded_bar(acc), (seed_phase >> acc) & 1u);
        seed_phase ^= 1u << acc;
        ptx::tc_fence_after();
        first = 0u;
      }
      if (FT && carrier) {
        // carrier tile: two UMMAs per k-step on the same A slab -- the data tile, and the tile-row's checksum product into
        // accumulator stage acc ^ 1 (a loop of its own: see the producer)
        const uint32_t c_tmem = tmem_base + (acc ^ 1) * BN;
        for (int kb = sg.kb_begin; kb < sg.kb_end; ++kb) {
          ptx::mbar_wait(full_bar(stage), phase);
          ptx::tc_fence_after();
          const uint32_t a_lo = desc_lo0 + static_cast<uint32_t>(stage) * (Cfg::kStageBytes >> 4);
          const uint32_t b_lo = a_lo + (Cfg::kABytes >> 4);
          const uint32_t e_lo = e_lo0 + static_cast<uint32_t>(stage) * (Cfg::kESlotBytes >> 4);
          const bool last_kb = (kb + 1 == sg.kb_end);
          if (ptx::elect_one()) {
#pragma unroll
            for (int j = 0; j < kBK / 8; ++j) {
              const uint64_t da = desc_hi | static_cast<uint64_t>(a_lo + j * kstep16);
              const uint64_t db = desc_hi | static_cast<uint64_t>(b_lo + j * kstep16);
              const uint64_t de = desc_hi | static_cast<uint64_t>(e_lo + j * kstep16);
              const uint32_t accum = (j == 0) ? (first ^ 1u) : 1u;
              if (CG == 2) {
                ptx::mma_tf32_cg2(d_tmem, da, db, idesc_t, accum);
                ptx::mma_tf32_cg2(c_tmem, da, de, idesc_c, accum);
              } else {
                ptx::mma_tf32(d_tmem, da, db, idesc_t, accum);
                ptx::mma_tf32(c_tmem, da, de, idesc_c, accum);
              }
            }
            if (CG == 2) ptx::mma_commit_cg2(empty_bar(stage), 0x3);
            else ptx::mma_commit(empty_bar(stage));
            if (last_kb) {
              if (CG == 2) ptx::mma_commit_cg2(tfull_bar(acc), 0x3);
              else ptx::mma_commit(tfull_bar(acc));
            }
          }
          __syncwarp();
          first = 0u;
          if (++stage == kStages) {
            stage = 0;
            phase ^= 1u;
          }
        }
      } else
      for (int kb = sg.kb_begin; kb < sg.kb_end; ++kb) {
        ptx::mbar_wait(full_bar(stage), phase);
        ptx::tc_fence_after();
        const uint32_t a_lo = desc_lo0 + static_cast<uint32_t>(stage) * (Cfg::kStageBytes >> 4);
        const uint32_t b_lo = a_lo + (Cfg::kABytes >> 4);
        const bool last_kb = (kb + 1 == sg.kb_end);
        if (ptx::elect_one()) {
#pragma unroll
          for (int j = 0; j < kBK / 8; ++j) {
            const uint64_t da = desc_hi | static_cast<uint64_t>(a_lo + j * kstep16);
            const uint64_t db = desc_hi | static_cast<uint64_t>(b_lo + j * kstep16);
            const uint32_t accum = (j == 0) ? (first ^ 1u) : 1u;
            if (CG == 2) ptx::mma_tf32_cg2(d_tmem, da, db, idesc_t, accum);
            else ptx::mma_tf32(d_tmem, da, db, idesc_t, accum);
          }
          // frees the smem slot (in both CTAs) once these MMAs have read it
          if (CG == 2) ptx::mma_commit_cg2(empty_bar(stage), 0x3);
          else ptx::mma_commit(empty_bar(stage));
          if (last_kb) {  // accumulator complete (both CTAs' epilogues)
            if (CG == 2) ptx::mma_commit_cg2(tfull_bar(acc), 0x3);
            else ptx::mma_commit(tfull_bar(acc));
          }
        }
        __syncwarp();
        first = 0u;
        if (++stage == kStages) {
          stage = 0;
          phase ^= 1u;
        }
      }
      if (p.trace != nullptr && lane == 0) trace_put(p, unit, item_idx, 3, globaltimer_ns());
      if (kAccStages == 2) {
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1u;
      } else {
        acc_phase ^= 1u;
      }
    }
  } else if (warp >= 4 && warp < 8) {
    // ===================================================================== epilogue (4 warps per CTA, lane = row)
    const int q = warp & 3;  // TMEM lane quadrant this warp may access
    const int row = q * 32 + lane;
    const uint32_t tempty_leader = (CG == 2) ? ptx::mapa(tempty_bar(0), 0) : tempty_bar(0);
    int acc = 0;
    uint32_t acc_phase = 0;
    SegIter it(p, unit);
    Segment sg;
    const size_t ws_slab = static_cast<size_t>(kBM) * BN;  // floats per (unit, CTA) partial tile
    int item_idx = -1;
    const bool tracer = p.trace != nullptr && is_leader && q == 0 && lane == 0;
    while (it.next(sg)) {
      ++item_idx;
      const TileCoord tc = decode_tile(p, sg.tile);
      const int m0_cta = (tc.m_blk * CG + static_cast<int>(cta_rank)) * kBM;
      const int n0 = (FT && tc.is_chk) ? tc.n_blk * chk_cols_per_tile(BN) : tc.n_blk * BN;
      const int m = m0_cta + row;
      ExpectedChk xp;
      xp.ready = false;
      if (FT && !tc.is_chk && (sg.kind == 0 || sg.kind == 2 || sg.kind == 6) && !(p.dbg_flags & 1)) {
        // poll the slab flag (at most ~2 polls per microsecond) until it is raised or the accumulator is complete
        try_prefetch_expected(p, q, lane, m, m0_cta, tc.n_blk, xp);
        while (!xp.ready && !ptx::mbar_try_wait(tfull_bar(acc), acc_phase)) {
          __nanosleep(400);
          try_prefetch_expected(p, q, lane, m, m0_cta, tc.n_blk, xp);
        }
      }
      ptx::mbar_wait(tfull_bar(acc), acc_phase);
      ptx::tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * BN;
      if (tracer) {
        trace_put(p, unit, item_idx, 4, globaltimer_ns());
        trace_put(p, unit, item_idx, 7, static_cast<unsigned long long>(sg.tile) | (static_cast<unsigned long long>(sg.kind) << 24));
      }

      if (FT && sg.kind == 6) {
        // carrier: publish the tile-row's expected checksums (accumulator stage acc ^ 1), raise the slab flag, hand the
        // stage back to the UMMA warp -- then this tile is checked like any other (its own flag is the last one to wait for)
        const uint32_t taddr_c = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + (acc ^ 1) * BN;
        store_tile<BN>(taddr_c, p.chk_out + m, m < p.M, 0, p.n_chk_cols, p.M, 1.0f, 0.0f, 0, (p.n_chk_cols + 31) / 32);
        __threadfence();
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          atomicExch(p.chk_flags + ((m0_cta >> 5) + q) * chk_flags_per_slab(p), p.chk_epoch);
          if (CG == 2) ptx::mbar_arrive_cluster(ptx::mapa(chk_drained_bar, 0));
          else ptx::mbar_arrive(chk_drained_bar);
        }
        __syncwarp();
      }
      const bool parks = sg.kind == 1 || sg.kind == 3;  // first / middle piece of a cut tile
      if (parks) {
        // park the raw sums of this piece for the unit that owns the next one
        const int slot = (sg.slice * p.sk_tiles + sg.split_idx) * CG + static_cast<int>(cta_rank);
        sk_dump_partial<BN>(p, taddr, p.sk_ws + slot * ws_slab + row, p.sk_flags + slot * 4 + q, lane);
      }
      if (parks) {
        // nothing to store yet
      } else if (FT && tc.is_chk) {
        // checksum tile-column: publish R = A * [e, w]^T for these 128 rows, then raise the slab flag
        const int n_hi = min(p.n_chk_cols, n0 + chk_cols_per_tile(BN));  // columns beyond belong to the next item
        store_tile<BN>(taddr, p.chk_out + static_cast<size_t>(tc.slice) * p.M * p.n_chk_cols + m, m < p.M, n0, n_hi, p.M, 1.0f, 0.0f, 0,
                       (n_hi - n0 + 31) / 32);
        __threadfence();
        __syncwarp();
        if (lane == 0)
          atomicExch(p.chk_flags + ((m0_cta >> 5) + q) * chk_flags_per_slab(p) + tc.slice * p.tiles_c + tc.n_blk, p.chk_epoch);
      } else {
        // final epilogue of a data tile; with epi_assist the helper warp of this quadrant owns the chunks [kMid, BN/32)
        const bool assist = p.epi_assist != 0 && BN >= 64;
        const int c_mid = assist ? kMid : BN / 32;
        int fix_col = -1;
        float fix_val = 0.0f;
        bool redo = false;
        float own_s1 = 0.0f;
        if (FT && !(p.dbg_flags & 1))
          abft_check<BN>(p, taddr, q, lane, m, m0_cta, n0, tc.n_blk, fix_col, fix_val, redo, xp, own_s1, c_mid, xchg_base(q), 4 + q);
        // rows to recompute are skipped by both store passes (the helper reads the mask after the pair barrier below)
        const unsigned redo_mask = FT ? __ballot_sync(0xffffffffu, redo) : 0u;
        // rows repaired in tensor memory: the sums of pass 1 no longer describe what a protected store pass re-reads
        const unsigned stale_mask = FT ? __ballot_sync(0xffffffffu, fix_col >= 0) : 0u;
        if (FT && assist && !(p.dbg_flags & 1) && lane == 0) {
          ptx::st_shared_u32(xchg_base(q), redo_mask);
          if constexpr (PROT) ptx::st_shared_u32(xchg_base(q) + 4, stale_mask);
        }
        if (tracer) trace_put(p, unit, item_idx, 5, globaltimer_ns());
        if (FT) {
          // rare: write the recomputed elements back into the accumulator (one lane = one row at a time, like the
          // injection path), so that the store pass stays free of per-element patching (a dynamically indexed patch of the
          // register tile had pushed it into local memory: 6.6 us instead of 3.6 us per tile)
          unsigned fix_mask = stale_mask;
          while (fix_mask != 0u) {
            const int src = __ffs(fix_mask) - 1;
            fix_mask &= fix_mask - 1u;
            const int col = __shfl_sync(0xffffffffu, fix_col, src);
            const float val = __shfl_sync(0xffffffffu, fix_val, src);
            uint32_t x = ptx::tmem_ld_x1(taddr + col);
            ptx::tmem_wait_ld();
            if (lane == src) x = f2u(val);
            ptx::tmem_st_x1(taddr + col, x);
            ptx::tmem_wait_st();
          }
          if (p.inject_mode == 2) inject_after_check<BN>(p, taddr, q, lane, m0_cta, n0);
        }
        if (assist && FT && !(p.dbg_flags & 1)) {  // corrections are in tensor memory: the helper may store its half
          ptx::tc_fence_before();
          ptx::named_bar_sync(4 + q, 64);
        }
        if (PROT && FT && !(p.dbg_flags & 1) && n0 + BN <= p.N) {
          uint32_t bad_bits = 0u;
          const int bad_col = stored_value_fault<BN>(p, q, lane, m0_cta, n0, 0, c_mid, bad_bits);
          protected_store_pass<BN>(taddr, p.A, p.B, p.C, p.lda, p.ldb, p.ldc, p.N, p.K, p.alpha, p.beta, p.stats,
                                   p.recompute != 0 && p.detect_only == 0, m, m0_cta + q * 32, m < p.M && !redo, n0, 0, c_mid, own_s1,
                                   ((stale_mask >> lane) & 1u) == 0u, bad_col, bad_bits, lane);
        } else {
          store_tile<BN>(taddr, p.C + m, m < p.M && !redo, n0, p.N, p.ldc, p.alpha, p.beta, 0, c_mid);
        }
        if (FT && redo_mask != 0u) {  // rare, warp-uniform: recompute the flagged rows from global memory
          unsigned rm = redo_mask;
          while (rm != 0u) {
            const int r = __ffs(rm) - 1;
            rm &= rm - 1u;
            recompute_row<BN>(p.A, p.B, p.C, p.lda, p.ldb, p.ldc, p.N, p.K, p.alpha, p.beta, m0_cta + q * 32 + r, n0, lane);
          }
        }
        if (assist) {  // both halves are out of tensor memory
          ptx::tc_fence_before();
          ptx::named_bar_sync(4 + q, 64);
        }
      }
      // release this accumulator stage back to the MMA warp (of the leader CTA)
      ptx::tc_fence_before();
      __syncwarp();
      if (tracer) trace_put(p, unit, item_idx, 6, globaltimer_ns());
      if (lane == 0) {
        if (CG == 2) ptx::mbar_arrive_cluster(tempty_leader + 8u * acc);
        else ptx::mbar_arrive(tempty_bar(acc));
        ptx::red_release_shared_add(epi_count, 1u);
      }
      if (kAccStages == 2) {
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1u;
      } else {
        acc_phase ^= 1u;
      }
    }
  }

  else if (warp >= 8) {
    // ===================================================================== helper warps (TMEM lane quadrant = warp & 3)
    const int q = warp & 3;
    if (p.sk_tiles > 0 || (p.epi_assist != 0 && BN >= 64)) {
      const uint32_t seeded_leader = (CG == 2) ? ptx::mapa(seeded_bar(0), 0) : seeded_bar(0);
      const size_t ws_slab = static_cast<size_t>(kBM) * BN;
      const int row = q * 32 + lane;
      const bool assist_on = p.epi_assist != 0 && BN >= 64;
      // The upper half of the final epilogue of item `a` (same structure as the epilogue warp's lower half: the barriers of
      // the pair must match one to one).
      auto assist = [&](const Segment &a, int a_acc, uint32_t a_phase) {
        if (!assist_on) return;
        // Observe EVERY item's accumulator-complete phase, assisted or not: a parity wait is only unambiguous within one
        // phase of the barrier, and a run of four parking / checksum items would otherwise put this warp two phases ahead.
        ptx::mbar_wait(tfull_bar(a_acc), a_phase);
        const bool parks = a.kind == 1 || a.kind == 3;
        if (parks) return;
        const TileCoord tc = decode_tile(p, a.tile);
        if (FT && tc.is_chk) return;
        ptx::tc_fence_after();
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + a_acc * BN;
        const int m0_cta = (tc.m_blk * CG + static_cast<int>(cta_rank)) * kBM;
        const int m = m0_cta + row;
        uint32_t skip = 0u, stale = 0u;
        float s1 = 0.0f, s2 = 0.0f, sabs = 0.0f;
        if (FT && !(p.dbg_flags & 1)) {
          if (p.inject_mode != 0) {
            ptx::named_bar_sync(4 + q, 64);  // injected
            ptx::tc_fence_after();
          }
          abft_row_sums<BN>(taddr, kMid, BN / 32, s1, s2, sabs);
          ptx::st_shared_u32(xchg_base(q) + lane * 12, f2u(s1));
          ptx::st_shared_u32(xchg_base(q) + lane * 12 + 4, f2u(s2));
          ptx::st_shared_u32(xchg_base(q) + lane * 12 + 8, f2u(sabs));
          ptx::named_bar_sync(4 + q, 64);  // partial sums handed over
          ptx::named_bar_sync(4 + q, 64);  // verdict reached, corrections written to tensor memory
          ptx::tc_fence_after();
          skip = (ptx::ld_acquire_shared_u32(xchg_base(q)) >> lane) & 1u;  // rows the epilogue warp recomputes
          if constexpr (PROT) stale = (ptx::ld_acquire_shared_u32(xchg_base(q) + 4) >> lane) & 1u;  // rows it repaired in tensor memory
        }
        const int n0 = tc.n_blk * BN;
        if (PROT && FT && !(p.dbg_flags & 1) && n0 + BN <= p.N) {
          uint32_t bad_bits = 0u;
          const int bad_col = stored_value_fault<BN>(p, q, lane, m0_cta, n0, kMid, BN / 32, bad_bits);
          protected_store_pass<BN>(taddr, p.A, p.B, p.C, p.lda, p.ldb, p.ldc, p.N, p.K, p.alpha, p.beta, p.stats,
                                   p.recompute != 0 && p.detect_only == 0, m, m0_cta + q * 32, m < p.M && !skip, n0, kMid, BN / 32, s1,
                                   stale == 0u, bad_col, bad_bits, lane);
        } else {
          store_tile<BN>(taddr, p.C + m, m < p.M && !skip, n0, p.N, p.ldc, p.alpha, p.beta, kMid, BN / 32);
        }
        ptx::tc_fence_before();
        ptx::named_bar_sync(4 + q, 64);  // both halves are out of tensor memory
      };
      int acc = 0;
      uint32_t acc_phase = 0;
      int item_idx = -1;
      int first_kind = 0;
      bool have_prev = false;
      Segment prev;
      int prev_acc = 0;
      uint32_t prev_phase = 0;
      SegIter it(p, unit);
      Segment sg;
      while (it.next(sg)) {
        ++item_idx;
        if (item_idx == 0) first_kind = sg.kind;
        if (sg.kind == 2 || sg.kind == 3) {
          // Seed first (it has to be in tensor memory before this item's first UMMA, i.e. during the previous item's main
          // loop), assist the previous item's epilogue afterwards.  The accumulator stage must have been drained by this
          // CTA's four epilogue warps (item_idx - 2 and before).  A parked accumulator never depends on a helper warp
          // (parking epilogues are not assisted), so waiting here for another unit's flag cannot close a cycle.
          // (after a carrier -- always item 0 -- stage 1 also holds the tile-row's checksum product until the carrier's
          //  epilogue has stored it: wait for that whole epilogue)
          if (item_idx >= 2 || (item_idx == 1 && first_kind == 6)) {
            const uint32_t need = item_idx >= 2 ? 4u * static_cast<uint32_t>(item_idx - 1) : 4u;
            ptx::Watchdog wd;
            while (ptx::ld_acquire_shared_u32(epi_count) < need) {
              __nanosleep(64);
              if (wd.tick()) break;
            }
          }
          ptx::tc_fence_after();
          const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * BN;
          const int slot = ((sg.slice - 1) * p.sk_tiles + sg.split_idx) * CG + static_cast<int>(cta_rank);
          sk_seed<BN>(p, taddr, p.sk_ws + slot * ws_slab + q * 32 + lane, p.sk_flags + slot * 4 + q, lane);
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if (CG == 2) ptx::mbar_arrive_cluster(seeded_leader + 8u * acc);
            else ptx::mbar_arrive(seeded_bar(acc));
          }
        }
        if (have_prev) assist(prev, prev_acc, prev_phase);
        prev = sg;
        prev_acc = acc;
        prev_phase = acc_phase;
        have_prev = true;
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1u;
      }
      if (have_prev) assist(prev, prev_acc, prev_phase);
    }
  }

  __syncwarp();  // reconverge the single-lane roles before the .aligned barriers below
  ptx::tc_fence_before();
  if (CG == 2) ptx::cluster_sync_all();  // no CTA may exit while its peer can still signal its barriers
  else __syncthreads();
  if (FT && p.peer_world > 0 && threadIdx.x == 0) {
    // fused verdict push: every CTA's counter updates are ordered before its arrival; the last arrival publishes
    __threadfence();
    const unsigned int arrived = atomicAdd(p.exit_count, 1u);
    if (arrived == gridDim.x - 1) {
      __threadfence();
      const volatile DeviceStats *st = p.stats;
      double v[8];
      v[0] = static_cast<double>(st->tiles);
      v[1] = static_cast<double>(st->rows_checked);
      v[2] = static_cast<double>(st->detected);
      v[3] = static_cast<double>(st->corrected);
      v[4] = static_cast<double>(st->uncorrectable);
      v[5] = static_cast<double>(st->checksum_faults);
      v[6] = static_cast<double>(__uint_as_float(st->max_abs_bits));
      v[7] = static_cast<double>(__uint_as_float(st->max_rel_bits));
      // every value travels with the launch's sequence number in ONE 16-byte store, so a reader can tell a complete
      // vector (eight equal sequence numbers) without a system-scope fence between data and flag: one NVLink round trip
      // at the end of the kernel instead of two
      for (int r = 0; r < p.peer_world; ++r) {
        double2 *slot = reinterpret_cast<double2 *>(p.peer_box[r] + p.peer_rank * kPeerSlotDoubles);
#pragma unroll
        for (int i = 0; i < 8; ++i) slot[i] = make_double2(v[i], p.peer_seq);
      }
      *p.exit_count = 0u;
    }
  }
  if (warp == 2) {
    ptx::tc_fence_after();
    if (CG == 2) ptx::tmem_dealloc_cg2(tmem_base, Cfg::kTmemCols);
    else ptx::tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------------------------
// Stand-alone encode pre-pass in front of the GEMM kernel (HBM-bound: it reads B once).  Four in-kernel alternatives
// were built and measured over two rounds -- helper warps reducing B stages from shared memory ("encoder tiles" /
// "encoder items"), and the idle warps of every CTA reducing B straight from global memory -- and removed: on an SM
// whose ingest port and shared-memory port are saturated by TMA + UMMA a second reader of B is starved (background
// loads ran 6x slower than on an idle SM), profiles/README.md.
// ------------------------------------------------------------------------------------------------------------
constexpr int kEncWarps = 8;

template <int BN, int KRQ, bool STREAM = false>
__global__ void __launch_bounds__(kEncWarps * 32, 2)
encode_b_kernel(const float *__restrict__ B, int N, int K, int ldb, float *__restrict__ chk, int chk_ld, int rounding,
                int tiles_n) {
  ptx::pdl_wait();               // (a programmatic dependent itself: the predecessor may still be reading the old vectors)
  ptx::pdl_launch_dependents();  // the GEMM kernel may start on SMs as they drain (its checksum items wait for this grid)
  encode_b_warp<BN, KRQ, STREAM>(B, N, K, ldb, chk, chk_ld, rounding, tiles_n, blockIdx.x * kEncWarps + (threadIdx.x >> 5),
                    gridDim.x * kEncWarps, threadIdx.x & 31);
}

}  // namespace ftsgemm
