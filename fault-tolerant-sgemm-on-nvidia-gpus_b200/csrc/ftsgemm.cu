// ftsgemm.cu -- host side of libftsgemm.so: the C ABI declared in include/ftsgemm.h.
//
// Owns: the kernel-variant table (reference: kernel/ft_sgemm/sgemm.cu:235-237 + code_gen/main.py:8-16), the id ->
// launch dispatch (reference: sgemm.cu:110-199, 256-430), TMA tensor-map construction, the encode pre-pass launch,
// the cuBLAS comparator rows (sgemm.cu:108,198,260), the non-fused ABFT baseline
// (include/baseline_ft_sgemm.cuh:1-33) and the device-side comparator (utils/utils.cu:61-77).
// There is NO CPU fallback: without an sm_100 device every compute entry point returns FTSGEMM_ERR_NO_DEVICE.
#include <cublas_v2.h>
#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdio>
#include <ctime>
#include <cstdlib>
#include <cstring>
#include <array>
#include <map>
#include <mutex>
#include <string>

#include "../../include/ftsgemm.h"
#include "ftsgemm_kernel.cuh"
#include "plan.h"

namespace {

using namespace ftsgemm;

// ------------------------------------------------------------------------------------------- variant table
struct Variant {
  ftsgemm_kernel_info info;
  int bn;  // CTA(-pair) tile N of the tcgen05 kernel (0 for library rows)
  int cg;  // 1 = one CTA per tile (UMMA M = 128), 2 = CTA pair per tile (cta_group::2, UMMA M = 256)
};

// Reference tiles from code_gen/main.py:8-16.  sm_100a tiles: UMMA M is 128 per CTA (256 for a CTA pair), so the
// reference's "tall" (128x32) and "huge" (128x128) shapes are literal; the four others map, in the reference's order of
// size, onto the remaining UMMA-legal shapes -- six names, six DISTINCT binaries (round 1 aliased small = tall and
// large = huge):   small 128x64   medium 256x64 (pair)   large 256x128 (pair)   tall 128x32   wide 128x256   huge 128x128.
// "giant" (ids 21/31) is the B200-only CTA-pair tile 256x256, "pair128" (22/32) an alias of large kept for round-1
// callers; ids 20 / 40 pick per shape (select_variant).  tile_k = K extent of one shared-memory stage (4 UMMA k-steps).
const Variant kVariants[] = {
    {{0, "cublas", 0, 0, 0, 0, 0, 0, 0, 0}, 0, 0},
    {{1, "kernel_sgemm_small", 0, 1, 16, 16, 16, 128, 64, 32}, 64, 1},
    {{2, "kernel_sgemm_medium", 0, 1, 32, 32, 8, 256, 64, 32}, 64, 2},
    {{3, "kernel_sgemm_large", 0, 1, 64, 64, 8, 256, 128, 32}, 128, 2},
    {{4, "kernel_sgemm_tall", 0, 1, 128, 32, 8, 128, 32, 32}, 32, 1},
    {{5, "kernel_sgemm_wide", 0, 1, 32, 128, 8, 128, 256, 32}, 256, 1},
    {{6, "kernel_sgemm_huge", 0, 1, 128, 128, 8, 128, 128, 32}, 128, 1},
    {{7, "cublas_tf32", 0, 0, 0, 0, 0, 0, 0, 0}, 0, 0},
    {{10, "abft_baseline", 1, 2, 0, 0, 256, 0, 0, 256}, 0, 0},
    {{11, "abft_kernel_small", 1, 1, 16, 16, 16, 128, 64, 32}, 64, 1},
    {{12, "abft_kernel_medium", 1, 1, 32, 32, 8, 256, 64, 32}, 64, 2},
    {{13, "abft_kernel_large", 1, 1, 64, 64, 8, 256, 128, 32}, 128, 2},
    {{14, "abft_kernel_tall", 1, 1, 128, 32, 8, 128, 32, 32}, 32, 1},
    {{15, "abft_kernel_wide", 1, 1, 32, 128, 8, 128, 256, 32}, 256, 1},
    {{16, "abft_kernel_huge", 1, 1, 128, 128, 8, 128, 128, 32}, 128, 1},
    {{20, "kernel_sgemm_auto", 0, 1, 0, 0, 0, 0, 0, 32}, 0, 0},
    {{21, "kernel_sgemm_giant", 0, 1, 0, 0, 0, 256, 256, 32}, 256, 2},
    {{22, "kernel_sgemm_pair128", 0, 1, 0, 0, 0, 256, 128, 32}, 128, 2},
    {{30, "abft_baseline_tf32", 1, 2, 0, 0, 256, 0, 0, 256}, 0, 0},
    {{31, "abft_kernel_giant", 1, 1, 0, 0, 0, 256, 256, 32}, 256, 2},
    {{32, "abft_kernel_pair128", 1, 1, 0, 0, 0, 256, 128, 32}, 128, 2},
    {{40, "abft_kernel_auto", 1, 1, 0, 0, 0, 0, 0, 32}, 0, 0},
};
constexpr int kNumVariants = sizeof(kVariants) / sizeof(kVariants[0]);

const Variant *find_variant(int id) {
  if (id == 8 || id == 9) id = 0;  // reference: ids outside the table run plain cuBLAS (sgemm.cu:197-199)
  for (int i = 0; i < kNumVariants; ++i)
    if (kVariants[i].info.id == id) return &kVariants[i];
  return nullptr;
}

// Per-shape choice of the tcgen05 variant (replaces the reference's manual id choice, sgemm.cu:110-199; SURVEY 8 f2).
// Measured on B200 (profiles/r02_sweep_small_all_variants.jsonl, r02_small_slices_*.jsonl; 20-launch bursts, us per
// launch): with few tiles the 74 CTA pairs are mostly idle with 256x256 tiles and the 256x128 pair tile ("large") is ahead --
//   plain: 1024^3 12.4 vs 17.0, 1536^3 16.4 vs 21.9, 2048^3 32.7 vs 27.8  -> giant from 49 tiles of 256x256 on;
//   ABFT:  1024^3 18.6 vs 22.2, 1536^3 33.8 vs 28.2                          -> giant from 25 tiles on.
int select_variant(int M, int N, bool ft) {
  const long long tiles256 = (static_cast<long long>(M) + 255) / 256 * ((static_cast<long long>(N) + 255) / 256);
  if (tiles256 >= (ft ? 25 : 49)) return ft ? FTSGEMM_ID_ABFT_GIANT : FTSGEMM_ID_SGEMM_GIANT;
  return ft ? FTSGEMM_ID_ABFT_LARGE : FTSGEMM_ID_SGEMM_LARGE;
}

// slab flags of the checksum tile-columns live in front of the expected-checksum matrix (one int per 32-row slab and
// checksum tile-column: 128 KiB for the 128 x 32 tile at 16384^2)
constexpr size_t kChkFlagBytes = 1u << 20;

// ------------------------------------------------------------------------------------------- debug knobs
std::mutex g_dbg_mu;
std::map<std::string, long long> g_dbg;
long long dbg(const char *key, long long dflt) {
  std::lock_guard<std::mutex> lk(g_dbg_mu);
  auto it = g_dbg.find(key);
  return it == g_dbg.end() ? dflt : it->second;
}

// ------------------------------------------------------------------------------------------- handle
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

}  // namespace

struct ftsgemm_handle_s {
  int device = 0;
  int num_sms = 0;
  cublasHandle_t cublas = nullptr;
  EncodeTiledFn encode_tiled = nullptr;
  DeviceStats *d_stats = nullptr;
  float *d_chk = nullptr;       // encoded checksum vectors [K][tiles_n*8]  (extra "rows" of B)
  size_t chk_bytes = 0;
  float *d_chk_out = nullptr;   // expected checksums M x (tiles_n*8), column-major, + slab flags behind it
  size_t chk_out_bytes = 0;
  const float *chk_for_b = nullptr;  // B pointer / shape the panel was encoded from
  int chk_n = 0, chk_k = 0, chk_bn = 0;
  // fused verdict exchange (ftsgemm_peer_*): this rank's mailbox (kMaxPeers slots), the peers' mailboxes mapped through
  // CUDA IPC, the exit counter of the publishing launches and their sequence number
  double *d_mailbox = nullptr;
  double *peer_box[kMaxPeers] = {};
  bool peer_opened[kMaxPeers] = {};
  int peer_world = 0, peer_rank = 0;
  unsigned long long peer_seq = 0;
  unsigned int *d_exit_count = nullptr;
  int *d_enc_done = nullptr;    // front-phase encode: warps done, monotonic over launches
  int enc_done_value = 0;
  float *d_lo = nullptr;        // 3xTF32: A_lo | B_lo
  size_t lo_bytes = 0;
  float *d_aux = nullptr;       // baseline vectors
  size_t aux_floats = 0;
  struct CachedPlan {
    std::vector<int> wave_target;   // per whole-tile ordinal: units that own more whole tiles than that
    int *d_wave_target = nullptr;
    ftsgemm::Plan plan;
    std::vector<int4> packed;   // host copy (kept alive for the async upload)
    int4 *d_items = nullptr;
    int *d_off = nullptr;
    bool uploaded = false;
  };
  std::map<std::array<long long, 6>, CachedPlan> plans;  // key: kernel id, M, N, K, units, forced slices
  int *d_wave_cnt = nullptr;    // wave re-synchronisation counters (cleared per launch)
  size_t wave_cnt_cap = 0;
  int chk_epoch = 0;
  float *d_sk = nullptr;        // split-K partial tiles + flags
  size_t sk_bytes = 0;
  int sk_epoch = 0;
  unsigned long long *d_trace = nullptr;  // debug timeline (ftsgemm_debug_trace), allocated on first use
  int trace_units = 0;
  float *d_stage[3] = {nullptr, nullptr, nullptr};  // run_host staging A, B, C
  size_t stage_bytes[3] = {0, 0, 0};
  cudaStream_t s_in = nullptr, s_out = nullptr;     // run_host: upload / download streams of the panel pipeline
  cudaEvent_t ev_in[16] = {}, ev_done[16] = {};
  double *d_verify = nullptr;   // {first_bad (as long long), num, den}
  std::map<int, int> max_units;     // per kernel instantiation (BN * 8 + FT * 4 + CG): co-resident CTAs / CTA pairs
  cudaStream_t last_stream = nullptr;
  unsigned long long launch_count = 0;  // kernels of THIS library launched through the handle (ftsgemm_launch_count)
  int last_cuda_error = 0;
  unsigned long long last_verify_bad = 0;
};

namespace {

#define FT_CUDA(h, call)                                   \
  do {                                                     \
    cudaError_t e__ = (call);                              \
    if (e__ != cudaSuccess) {                              \
      if (h) (h)->last_cuda_error = static_cast<int>(e__); \
      return FTSGEMM_ERR_CUDA;                             \
    }                                                      \
  } while (0)

#define FT_CUBLAS(h, call)                                 \
  do {                                                     \
    cublasStatus_t s__ = (call);                           \
    if (s__ != CUBLAS_STATUS_SUCCESS) {                    \
      if (h) (h)->last_cuda_error = static_cast<int>(s__); \
      return FTSGEMM_ERR_CUBLAS;                           \
    }                                                      \
  } while (0)

// Every entry point runs on the device the handle was created on, whatever the caller's current device is.
struct DeviceGuard {
  int prev = -1;
  bool switched = false;
  explicit DeviceGuard(ftsgemm_handle_t h) {
    if (h && cudaGetDevice(&prev) == cudaSuccess && prev != h->device) switched = cudaSetDevice(h->device) == cudaSuccess;
  }
  ~DeviceGuard() {
    if (switched) cudaSetDevice(prev);
  }
};

// The kernels' watchdog (ptx.cuh) raises a device-wide flag instead of trapping; reported once, then cleared.
int check_abort_flag(ftsgemm_handle_t h) {
  int flag = 0;
  FT_CUDA(h, cudaMemcpyFromSymbol(&flag, ptx::g_abort_flag, sizeof(int)));
  if (flag == 0) return FTSGEMM_OK;
  flag = 0;
  FT_CUDA(h, cudaMemcpyToSymbol(ptx::g_abort_flag, &flag, sizeof(int)));
  return FTSGEMM_ERR_TIMEOUT;
}

int make_tmap_2d(ftsgemm_handle_t h, CUtensorMap *tm, const float *base, uint64_t inner, uint64_t outer,
                 uint64_t ld_elems, uint32_t box_inner, uint32_t box_outer) {
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {ld_elems * sizeof(float)};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  const CUtensorMapSwizzle sw =
      static_cast<CUtensorMapSwizzle>(dbg("tma_swizzle", static_cast<long long>(CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B)));
  CUresult r = h->encode_tiled(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float *>(base), dims, strides, box,
                               estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    h->last_cuda_error = static_cast<int>(r);
    return FTSGEMM_ERR_CUDA;
  }
  return FTSGEMM_OK;
}

// 3-D view {32, K, rows/32} of a column-major rows x K operand (rows % 32 == 0): element (i, k, a) = base[(a*32+i) + k*ld].
// One box {32, kBK, atoms} lands in shared memory as [atom][k][32 floats] -- exactly the canonical MN-major layout the
// UMMA descriptors describe -- with a single TMA instruction.
int make_tmap_3d(ftsgemm_handle_t h, CUtensorMap *tm, const float *base, uint64_t rows, uint64_t kdim, uint64_t ld_elems,
                 uint32_t atoms_per_box) {
  cuuint64_t dims[3] = {kAtomMN, kdim, rows / kAtomMN};
  cuuint64_t strides[2] = {ld_elems * sizeof(float), kAtomMN * sizeof(float)};
  cuuint32_t box[3] = {kAtomMN, kBK, atoms_per_box};
  cuuint32_t estr[3] = {1, 1, 1};
  const CUtensorMapSwizzle sw =
      static_cast<CUtensorMapSwizzle>(dbg("tma_swizzle", static_cast<long long>(CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B)));
  CUresult r = h->encode_tiled(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float *>(base), dims, strides, box,
                               estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    h->last_cuda_error = static_cast<int>(r);
    return FTSGEMM_ERR_CUDA;
  }
  return FTSGEMM_OK;
}

// Largest grid (in work units = CTAs or CTA pairs) of this instantiation whose CTAs are all resident at once.  The
// persistent kernel's inter-CTA waits (checksum flags, parked accumulators, wave counters) are only deadlock-free for
// such a grid, so the planner never gets more units than this -- on a device partition (MPS active-thread percentage,
// green context) that is fewer than multiProcessorCount / CG.  Cached per handle (= per device).
template <int BN, bool FT, int CG, bool PROT = false>
int query_max_units(ftsgemm_handle_t h, int *out) {
  using Cfg = TileCfg<BN, FT, CG>;
  const int key = BN * 16 + (PROT ? 8 : 0) + (FT ? 4 : 0) + CG;
  auto it = h->max_units.find(key);
  if (it != h->max_units.end()) {
    *out = it->second;
    return FTSGEMM_OK;
  }
  auto kern = ftsgemm_tc_kernel<BN, FT, CG, PROT>;
  FT_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
  int units = 0;
  if (CG > 1) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(h->num_sms / CG * CG);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = Cfg::kSmemBytes;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CG;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    FT_CUDA(h, cudaOccupancyMaxActiveClusters(&units, kern, &cfg));
  } else {
    int per_sm = 0;
    FT_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kThreads, Cfg::kSmemBytes));
    units = (per_sm > 0 ? 1 : 0) * h->num_sms;  // one persistent CTA per SM
  }
  if (units > h->num_sms / CG) units = h->num_sms / CG;
  h->max_units[key] = units;
  *out = units;
  return FTSGEMM_OK;
}

template <int BN, bool FT, int CG, bool PROT = false>
int launch_tc(ftsgemm_handle_t h, const CUtensorMap &tmA, const CUtensorMap &tmB, const CUtensorMap &tmC,
              const KernelParams &p, int units, cudaStream_t stream) {
  // p.pdl_wait: the launch may overlap the tail of its predecessor in the stream (KernelParams::pdl_wait)
  using Cfg = TileCfg<BN, FT, CG>;
  auto kern = ftsgemm_tc_kernel<BN, FT, CG, PROT>;
  int resident = 0;
  const int qrc = query_max_units<BN, FT, CG, PROT>(h, &resident);  // (also sets the shared-memory attribute, once per handle)
  if (qrc) return qrc;
  if (units > resident) return FTSGEMM_ERR_UNSUPPORTED;  // the plan was built for more units than can be co-resident
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(units * CG);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = Cfg::kSmemBytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (CG > 1) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = CG;
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = 1;
    ++na;
  }
  if (p.pdl_wait) {
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  FT_CUDA(h, cudaLaunchKernelEx(&cfg, kern, tmA, tmB, tmC, p));
  return FTSGEMM_OK;
}

// Planner input for one launch (tile grid already set by plan_tiles).
// Measured on B200 (device timeline, profiles/r01_trace_*): a checksum tile's main loop takes 0.57-0.58 of a data tile's
// whatever its UMMA N (it is bound by the A-operand feed, L2 -> shared memory), one k-block of a 256x256 CTA-pair tile
// takes ~0.33 us, an item costs ~1.5 us of pipeline fill + drain, and a parked accumulator is back in the next owner's
// tensor memory ~8 us after the piece's last UMMA.
template <int BNv, int CGv>
void chk_costs(const KernelParams &p, double floor_cost, std::vector<double> *out) {
  for (int c = 0; c < p.tiles_c; ++c)
    out->push_back(std::max(floor_cost, static_cast<double>(chk_tile_width<BNv, CGv>(p, c)) / BNv));
}

int carrier_tile_index(const KernelParams &p, int m_blk);

PlanInput make_plan_input(int max_units, int CG, int BN, int K, const KernelParams &p) {
  PlanInput in;
  long long units = dbg("grid", 0);
  in.units = (units > 0 && units <= max_units) ? static_cast<int>(units) : max_units;
  in.chk_slices = p.chk_slices > 1 ? p.chk_slices : 1;
  in.n_chk_tiles = p.chk_in_carriers ? 0 : p.tiles_c * p.tiles_m * in.chk_slices;
  if (p.chk_in_carriers) {
    for (int m = 0; m < p.tiles_m; ++m) in.carriers.push_back(carrier_tile_index(p, m));
    in.carrier_cost = static_cast<double>(dbg("carrier_cost_permille", 1400)) * 1e-3;
  }
  in.n_data_tiles = p.tiles_m * p.tiles_n;
  in.num_kb = (K + kBK - 1) / kBK;
  in.tiles_m = p.tiles_m;
  // operands larger than ~3/4 of the 126 MB L2: keep the units in k-lockstep (plan.h)
  const long long lock = dbg("lockstep", -2);
  in.lockstep = lock >= 0 ? static_cast<int>(lock)
                          : (4.0 * K * (static_cast<double>(p.M) + p.N) > 96.0 * 1024 * 1024 ? 1 : 0);
  // a checksum item's main loop runs at 0.22 us per k-block whatever the size (round 2 timelines: 0.67-0.69 of a data
  // tile at 2048 .. 4096, where data tiles take 0.33 us per k-block out of L2; 0.58 where they are HBM-bound)
  const double chk_floor = static_cast<double>(dbg("chk_cost_permille", in.lockstep ? 580 : 680)) * 1e-3;
  if (BN == 32) chk_costs<32, 1>(p, chk_floor, &in.chk_col_cost);
  else if (BN == 64 && CG == 1) chk_costs<64, 1>(p, chk_floor, &in.chk_col_cost);
  else if (BN == 64) chk_costs<64, 2>(p, chk_floor, &in.chk_col_cost);
  else if (BN == 128 && CG == 1) chk_costs<128, 1>(p, chk_floor, &in.chk_col_cost);
  else if (BN == 128) chk_costs<128, 2>(p, chk_floor, &in.chk_col_cost);
  else if (CG == 1) chk_costs<256, 1>(p, chk_floor, &in.chk_col_cost);
  else chk_costs<256, 2>(p, chk_floor, &in.chk_col_cost);
  const double tile_us = in.num_kb * 0.333 * (static_cast<double>(BN) * CG / 512.0 < 0.25 ? 0.25 : static_cast<double>(BN) * CG / 512.0);
  in.item_overhead = static_cast<double>(dbg("item_overhead_ns", 1500)) * 1e-3 / tile_us;
  in.park_latency = static_cast<double>(dbg("park_latency_ns", 8000)) * 1e-3 / tile_us;
  in.seed_overhead = static_cast<double>(dbg("seed_overhead_ns", 2000)) * 1e-3 / tile_us;
  const long long force = dbg("splitk", -2);  // -2 auto, 0 off, s > 1: force s equal pieces
  in.max_slices = force == 0 ? 1 : 2;
  in.force_slices = force > 1 ? static_cast<int>(force) : 0;
  in.slab_bytes = static_cast<size_t>(CG) * kBM * BN * sizeof(float);
  in.full_search = dbg("plan_full_search", 0) != 0 ? 1 : 0;
  return in;
}

// Carrier tiles or checksum items?  Legal when the whole checksum-operand box fits the 4 KiB slot of a stage
// (n_chk_cols <= 32 * CG, i.e. N <= 4096 with 256-wide pair tiles), every operand goes through 3-D tensor maps and there is
// at most one carrier per unit (a carrier must be the FIRST item of its unit: tensor-memory stage 1 is only free then).
// Measured (profiles/r02_carriers_on_off.jsonl, us per launch, carriers vs checksum items): a carrier's main loop takes 1.39
// tile-times (59.8 vs 42.9 us at 4096^3) against 0.68 + epilogue for a checksum item, but it is a longer CHAIN: with fewer
// than ~2.3 waves of tiles the carrier + its unit's next tile set the makespan -- 2304^3 58.4 vs 53.8, 2560^3 67.5 vs 60.5,
// then 3328^3 111.9 vs 113.3, 3584^3 137.4 vs 144.8, 3840^3 172.0 vs 171.9, 4096^3 199.8 vs 202.3.
bool use_carriers(const KernelParams &p, int units, int CG) {
  const long long c = dbg("carriers", -2);
  if (c == 0) return false;
  const bool legal = p.tiles_c == 1 && p.n_chk_cols <= kAtomMN * CG && (p.tma3d & 7) == 7 && p.tiles_m <= units;
  if (!legal) return false;
  if (c > 0) return true;
  return 4ll * p.tiles_m * p.tiles_n >= 9ll * units;  // from 2.25 waves of data tiles on
}

// raster index (among the data tiles) of tile (m_blk, n_blk = 0): inverse of decode_tile
int carrier_tile_index(const KernelParams &p, int m_blk) {
  const int gsz = p.group_n < p.tiles_n ? p.group_n : p.tiles_n;
  return m_blk * gsz;
}

// K-slices of the checksum items (KernelParams::chk_slices): only where units would otherwise idle -- all data tiles and
// all slices run concurrently in one wave -- and a slice keeps at least 8 k-blocks.  Measured at 1024^3 (id 13): the
// checksum item's K loop (7 us, after the encode) + its epilogue were the critical path of a 19.5 us step.
int choose_chk_slices(const KernelParams &p, int units, int K) {
  const long long forced = dbg("chk_slices", -2);
  const int num_kb = (K + kBK - 1) / kBK;
  if (p.tiles_c != 1) return 1;
  int s = 1;
  if (forced >= 1) s = static_cast<int>(forced);
  else {
    const int spare = units - p.tiles_m * p.tiles_n;
    if (spare >= 2 * p.tiles_m) s = spare / p.tiles_m;
    if (s > 4) s = 4;
  }
  while (s > 1 && num_kb / s < 8) --s;
  return s < 1 ? 1 : s;
}

void plan_tiles(int M, int N, int BN, int CG, bool ft, KernelParams *p) {
  p->tiles_m = (M + kBM * CG - 1) / (kBM * CG);
  p->tiles_n = (N + BN - 1) / BN;
  long long g = dbg("group_n", 0);
  p->group_n = g > 0 ? static_cast<int>(g) : (2048 / BN > 0 ? 2048 / BN : 1);
  if (p->group_n > p->tiles_n) p->group_n = p->tiles_n;
  p->n_chk_cols = 0;
  p->tiles_c = 0;
  if (ft) {
    p->n_chk_cols = p->tiles_n * kChkPerTile;
    const int cw = chk_cols_per_tile(BN);
    p->tiles_c = (p->n_chk_cols + cw - 1) / cw;
    if (dbg("ft_dbg", 0) & 2) p->tiles_c = 0;  // experiment: no checksum tile-columns (expected checksums are garbage)
  }
}

int ensure_buf(ftsgemm_handle_t h, float **buf, size_t *have, size_t bytes) {
  if (*have >= bytes) return FTSGEMM_OK;
  if (*buf) FT_CUDA(h, cudaFree(*buf));
  *buf = nullptr;
  *have = 0;
  FT_CUDA(h, cudaMalloc(buf, bytes));
  *have = bytes;
  return FTSGEMM_OK;
}

int run_tc(ftsgemm_handle_t h, const Variant &v, int M, int N, int K, const float *dA, const float *dB, float *dC,
           float alpha, float beta, const ftsgemm_opts &o, cudaStream_t stream) {
  const int BN = v.bn, CG = v.cg;
  const bool ft = v.info.fault_tolerant != 0;
  if ((M % 4) || (N % 4)) return FTSGEMM_ERR_UNSUPPORTED;  // TMA global strides must be multiples of 16 bytes
  // work-plan items carry k-block indices in 16 bits and tile indices in 31; the trace / wave tables are sized per unit
  if ((K + kBK - 1) / kBK > 65535) return FTSGEMM_ERR_UNSUPPORTED;
  if ((static_cast<long long>(M + kBM * CG - 1) / (kBM * CG)) * ((N + BN - 1) / BN) > (1ll << 28)) return FTSGEMM_ERR_UNSUPPORTED;
  if ((reinterpret_cast<uintptr_t>(dA) | reinterpret_cast<uintptr_t>(dB) | reinterpret_cast<uintptr_t>(dC)) & 15)
    return FTSGEMM_ERR_INVALID_ARG;

  KernelParams p;
  memset(&p, 0, sizeof(p));
  p.M = M; p.N = N; p.K = K;
  p.C = dC; p.ldc = M;
  p.alpha = alpha; p.beta = beta;
  plan_tiles(M, N, BN, CG, ft, &p);
  // MN-major fp32 operands: 128B swizzle with 32B atoms.  One TMA box = 32 (M|N) x 32 (K) floats = 32 rows of
  // 128 bytes, so successive M|N atoms are kBK*128 bytes apart (LBO), successive groups of 4 K-rows 512 bytes (SBO),
  // and one UMMA k-step (8 K-rows) advances the start address by 1024 bytes.
  p.lbo_bytes = static_cast<unsigned>(dbg("lbo", kBK * 128));
  p.sbo_bytes = static_cast<unsigned>(dbg("sbo", 512));
  p.layout_type = static_cast<unsigned>(dbg("layout_type", 1));
  p.kstep_bytes = static_cast<unsigned>(dbg("kstep", 1024));
  p.tau_abs = o.tau_abs > 0 ? o.tau_abs : 1e-3f;
  p.tau_rel = o.tau_rel > 0 ? o.tau_rel : 1e-5f;  // 13x the measured fault-free floor at K = 8192 (7.6e-7)
  p.detect_only = o.detect_only;
  p.recompute = o.no_recompute ? 0 : 1;
  p.A = dA;
  p.B = dB;
  p.lda = M;
  p.ldb = N;
  p.inject_mode = ft ? o.inject_mode : 0;
  p.selftest_value = o.selftest_value;
  p.selftest_row = o.selftest_row & (kBM - 1);  // (>= 0: validated by load_opts)
  p.selftest_col = o.selftest_col % BN;
  p.n_faults = o.n_faults < 0 ? 0 : (o.n_faults > kMaxFaults ? kMaxFaults : o.n_faults);
  for (int i = 0; i < p.n_faults; ++i) {
    p.faults[i].row = o.faults[i].row;
    p.faults[i].col = o.faults[i].col;
    p.faults[i].mode = o.faults[i].mode;
    p.faults[i].add_value = o.faults[i].add_value;
    p.faults[i].xor_mask = o.faults[i].xor_mask;
  }
  p.stats = h->d_stats;
  if (ft && h->peer_world > 0) {  // fused verdict push to every rank's mailbox
    for (int r = 0; r < h->peer_world; ++r) p.peer_box[r] = h->peer_box[r];
    p.peer_world = h->peer_world;
    p.peer_rank = h->peer_rank;
    p.peer_seq = static_cast<double>(++h->peer_seq);
    p.exit_count = h->d_exit_count;
  }

  CUtensorMap tmA, tmB, tmC;
  bool enc_front = false;
  const bool allow3d = dbg("tma3d", 1) != 0;
  int rc;
  if (allow3d && M % kAtomMN == 0) {
    rc = make_tmap_3d(h, &tmA, dA, M, K, M, kBM / kAtomMN);
    p.tma3d |= 1;
  } else {
    rc = make_tmap_2d(h, &tmA, dA, M, K, M, kAtomMN, kBK);
  }
  if (rc) return rc;
  if (allow3d && N % kAtomMN == 0) {
    rc = make_tmap_3d(h, &tmB, dB, N, K, N, BN / CG / kAtomMN);
    p.tma3d |= 2;
  } else {
    rc = make_tmap_2d(h, &tmB, dB, N, K, N, kAtomMN, kBK);
  }
  if (rc) return rc;
  tmC = tmB;
  if (ft) {
    // checksum vectors of B: 8 columns per N-tile, appended to B as extra tile-columns of the same GEMM
    p.dbg_flags = static_cast<int>(dbg("ft_dbg", 0)) & 1;
    const int chk_ld = (p.n_chk_cols + kAtomMN - 1) / kAtomMN * kAtomMN;  // padded so the 3-D TMA view is exact; pad
                                                                          // columns are never stored (n_chk_cols mask)
    const int n_slabs = p.tiles_m * CG * (kBM / 32);
    const float *chk_before = h->d_chk;
    rc = ensure_buf(h, &h->d_chk, &h->chk_bytes, static_cast<size_t>(K) * chk_ld * sizeof(float));
    if (rc) return rc;
    if (h->d_chk != chk_before) h->chk_for_b = nullptr;  // reallocated: the cached encode is gone
    const size_t out_floats = static_cast<size_t>(M) * p.n_chk_cols;
    const size_t n_flags = static_cast<size_t>(n_slabs) * p.tiles_c;
    const float *out_before = h->d_chk_out;
    rc = ensure_buf(h, &h->d_chk_out, &h->chk_out_bytes, kChkFlagBytes + out_floats * sizeof(float));
    if (rc) return rc;
    if (n_flags * sizeof(int) > kChkFlagBytes) return FTSGEMM_ERR_UNSUPPORTED;
    p.chk_flags = reinterpret_cast<int *>(h->d_chk_out);  // fixed location: stale flags never equal a new epoch
    p.chk_out = h->d_chk_out + kChkFlagBytes / sizeof(float);
    if (h->d_chk_out != out_before || h->chk_epoch > (1 << 30)) {
      FT_CUDA(h, cudaMemsetAsync(p.chk_flags, 0, kChkFlagBytes, stream));
      h->chk_epoch = 0;
    }
    p.chk_epoch = ++h->chk_epoch;
    p.dbg_flags = static_cast<int>(dbg("ft_dbg", 0)) & 1;
    const bool reuse = o.reuse_b_checksums && h->chk_for_b == dB && h->chk_n == N && h->chk_k == K && h->chk_bn == BN;
    // Default: the encode is a FRONT PHASE of the GEMM kernel (KernelParams::enc_front) -- one launch per fused GEMM, like
    // the reference (sgemm.cu:191-192).  Measured equal to the stand-alone pre-pass within noise from 2048^3 to 12288^3
    // (profiles/r02_front_phase_vs_prepass.jsonl: 200.0 vs 200.6 us at 4096^3, 1437 vs 1442 at 8192^3, -2.6 us at 2560^3);
    // only below ~8 MB of B (1024^3: 23.0 vs 22.1 us) the two-launch form is kept.
    const long long ef = dbg("enc_front", -2);
    enc_front = !reuse && (ef >= 0 ? ef != 0 : 4.0 * N * static_cast<double>(K) >= static_cast<double>(dbg("enc_front_min_mb", 8)) * 1048576.0);
    if (enc_front) {
      p.enc_front = 1;
      p.enc_out = h->d_chk;
      p.enc_ld = chk_ld;
    }
    if (!reuse && !enc_front) {
      // stand-alone pre-pass in the caller's stream
      const int rounding = static_cast<int>(dbg("enc_rounding", 0));
      // grid-stride over (column block, k-row group) items.  Item size (8 / 4 KiB) and grid (2 / 4 blocks per SM) make no
      // measurable difference (profiles/r01_probe22_*: 695-698 TFLOP/s at 4096^3 for all four): the pass is HBM time.
      const int grid = static_cast<int>(dbg("enc_blocks_per_sm", 4)) * h->num_sms;
      const bool small_items = dbg("enc_kr", 8) == 4;
      const bool chain = dbg("pdl_chain", 1) != 0;
      // B larger than ~half of L2: read it with evict-first loads (it cannot stay resident for the GEMM anyway)
      const long long sb = dbg("enc_stream", -2);
      const bool stream_b = sb > 0;  // measured at 8192^3: 1550 vs 1480 us per step -- the tail of B the pre-pass leaves in L2 is
                                     // worth more to the GEMM's first wave than the residue it evicts: off by default
#define FT_ENC(bn)                                                                                                          \
  if (BN == bn) {                                                                                                           \
    cudaLaunchConfig_t ec = {};                                                                                             \
    ec.gridDim = dim3(grid);                                                                                                \
    ec.blockDim = dim3(kEncWarps * 32);                                                                                     \
    ec.stream = stream;                                                                                                     \
    cudaLaunchAttribute ea[1];                                                                                              \
    ea[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;                                                          \
    ea[0].val.programmaticStreamSerializationAllowed = 1;                                                                   \
    ec.attrs = ea;                                                                                                          \
    ec.numAttrs = chain ? 1 : 0;                                                                                            \
    const float *eb = dB;                                                                                                   \
    float *eo = h->d_chk;                                                                                                   \
    int en = N, ek = K, el = chk_ld, er = rounding, et = p.tiles_n;                                                         \
    if (small_items) FT_CUDA(h, cudaLaunchKernelEx(&ec, encode_b_kernel<bn, 4, false>, eb, en, ek, en, eo, el, er, et));    \
    else if (stream_b) FT_CUDA(h, cudaLaunchKernelEx(&ec, encode_b_kernel<bn, 8, true>, eb, en, ek, en, eo, el, er, et));   \
    else FT_CUDA(h, cudaLaunchKernelEx(&ec, encode_b_kernel<bn, 8, false>, eb, en, ek, en, eo, el, er, et));                \
  }
      FT_ENC(32) FT_ENC(64) FT_ENC(128) FT_ENC(256)
      ++h->launch_count;
#undef FT_ENC
      FT_CUDA(h, cudaGetLastError());
      // The GEMM launch below becomes a programmatic dependent of this kernel: its CTAs start on SMs as they drain, and
      // only its checksum items wait for the pre-pass to complete.  Measured: +7.8 % at 2048^3, +1.2 % at 4096^3, but
      // -1.4 % at 8192^3 (CTAs that start early fall out of k-lockstep with the others), hence the size limit.
      const long long pdl = dbg("pdl", -2);
      p.pdl_wait = pdl >= 0 ? (pdl != 0) : (4.0 * K * (static_cast<double>(M) + N) <= 160.0 * 1024 * 1024);
    }
    if (!reuse) { h->chk_for_b = dB; h->chk_n = N; h->chk_k = K; h->chk_bn = BN; }
    p.chk_box_bytes = BN / CG * kBK * static_cast<int>(sizeof(float));
    if (allow3d) {
      // the checksum operand's box only spans the atoms that exist (e.g. 128 of 256 columns at N = 8192), so a
      // checksum item moves A plus a small B box per stage
      int atoms = BN / CG / kAtomMN;
      if (p.tiles_c == 1) {
        const int w = (p.n_chk_cols + 32 * CG - 1) / (32 * CG) * (32 * CG);
        atoms = (w < BN ? w : BN) / CG / kAtomMN;
      }
      p.chk_box_bytes = atoms * kAtomMN * kBK * static_cast<int>(sizeof(float));
      rc = make_tmap_3d(h, &tmC, h->d_chk, chk_ld, K, chk_ld, atoms);
      p.tma3d |= 4;
    } else {
      rc = make_tmap_2d(h, &tmC, h->d_chk, chk_ld, K, chk_ld, kAtomMN, kBK);
    }
    if (rc) return rc;
  }
  // ---- work plan (plan.h), cached per shape on the handle
  int max_units = 0;
  {
    int qrc = FTSGEMM_ERR_UNSUPPORTED;
#define FT_QUERY(bn, cg) \
  if (BN == bn && CG == cg) qrc = ft ? query_max_units<bn, true, cg>(h, &max_units) : query_max_units<bn, false, cg>(h, &max_units);
    FT_QUERY(32, 1) FT_QUERY(64, 1) FT_QUERY(128, 1) FT_QUERY(256, 1) FT_QUERY(64, 2) FT_QUERY(128, 2) FT_QUERY(256, 2)
#undef FT_QUERY
    if (qrc) return qrc;
    if (max_units < 1) return FTSGEMM_ERR_UNSUPPORTED;  // not a single CTA (pair) of this kernel fits on the device partition
  }
  if (ft) {
    // Carrier tiles instead of checksum items (KernelParams::chk_in_carriers, use_carriers)
    p.chk_in_carriers = use_carriers(p, max_units, CG) ? 1 : 0;
    p.chk_slices = p.chk_in_carriers ? 1 : choose_chk_slices(p, max_units, K);
    const size_t n_flags_s = static_cast<size_t>(p.tiles_m) * CG * (kBM / 32) * p.tiles_c * p.chk_slices;
    if (p.chk_slices > 1 && n_flags_s * sizeof(int) > kChkFlagBytes) p.chk_slices = 1;
    // Default tau_rel beyond K = 8192 (DESIGN.md section 5): with non-negative operands the accumulator's truncation-like
    // rounding adds up with K instead of cancelling, so the fault-free residual grows like K: 1e-5 * K / 8192.  Checksum
    // K-slices restart the expected checksum's accumulation and the data row's rounding no longer cancels against it:
    // 2.5e-8 * K (measured U[0,1) operands, (1024, 1024, K): 5.2e-9 * K; K = 16384 .. 65536 were all flagged at 1e-5).
    if (!(o.tau_rel > 0))
      p.tau_rel = fmaxf(1e-5f, (p.chk_slices > 1 ? 2.5e-8f : 1e-5f / 8192.0f) * static_cast<float>(K));
    if (p.chk_slices > 1) {
      // one plane of expected checksums per slice
      const size_t out_floats = static_cast<size_t>(M) * p.n_chk_cols * p.chk_slices;
      const float *out_before = h->d_chk_out;
      rc = ensure_buf(h, &h->d_chk_out, &h->chk_out_bytes, kChkFlagBytes + out_floats * sizeof(float));
      if (rc) return rc;
      if (h->d_chk_out != out_before) {  // reallocated: fresh flags, restart the epoch
        FT_CUDA(h, cudaMemsetAsync(h->d_chk_out, 0, kChkFlagBytes, stream));
        h->chk_epoch = 1;
        p.chk_epoch = 1;
      }
      p.chk_flags = reinterpret_cast<int *>(h->d_chk_out);
      p.chk_out = h->d_chk_out + kChkFlagBytes / sizeof(float);
    }
  }
  const PlanInput pin = make_plan_input(max_units, CG, BN, K, p);
  const std::array<long long, 6> key = {v.info.id, M, N, K, pin.units,
                                        pin.force_slices * 16 + pin.max_slices + pin.lockstep * 8192 + pin.full_search * 16384 + pin.chk_slices * 65536 + (p.chk_in_carriers ? 1048576 : 0)};
  ftsgemm_handle_s::CachedPlan &cp = h->plans[key];
  if (!cp.uploaded) {
    if (h->plans.size() > 64) {  // bound the cache: drop everything but this entry
      for (auto it = h->plans.begin(); it != h->plans.end();) {
        if (&it->second == &cp) { ++it; continue; }
        cudaFree(it->second.d_items);
        cudaFree(it->second.d_off);
        cudaFree(it->second.d_wave_target);
        it = h->plans.erase(it);
      }
    }
    cp.plan = build_plan(pin);
    cp.packed.resize(cp.plan.items.size());
    for (size_t i = 0; i < cp.plan.items.size(); ++i) {
      const PlanItem &it = cp.plan.items[i];
      cp.packed[i] = make_int4(it.tile, it.kb_begin | (it.kb_end << 16), it.kind | (it.slice << 8), it.split_idx);
    }
    FT_CUDA(h, cudaMalloc(&cp.d_items, std::max<size_t>(1, cp.packed.size()) * sizeof(int4)));
    FT_CUDA(h, cudaMalloc(&cp.d_off, cp.plan.offsets.size() * sizeof(int)));
    FT_CUDA(h, cudaMemcpyAsync(cp.d_items, cp.packed.data(), cp.packed.size() * sizeof(int4), cudaMemcpyHostToDevice, stream));
    FT_CUDA(h, cudaMemcpyAsync(cp.d_off, cp.plan.offsets.data(), cp.plan.offsets.size() * sizeof(int), cudaMemcpyHostToDevice, stream));
    {  // wave targets (see KernelParams::wave_cnt)
      std::vector<int> per_unit(static_cast<size_t>(cp.plan.units), 0);
      int max_w = 0;
      for (int u = 0; u < cp.plan.units; ++u) {
        for (int i = cp.plan.offsets[u]; i < cp.plan.offsets[u + 1]; ++i)
          if (cp.plan.items[i].kind == 0 && cp.plan.items[i].tile >= pin.n_chk_tiles) ++per_unit[u];
        max_w = std::max(max_w, per_unit[u]);
      }
      cp.wave_target.assign(static_cast<size_t>(max_w) + 1, 0);
      for (int u = 0; u < cp.plan.units; ++u)
        for (int w = 0; w < per_unit[u]; ++w) ++cp.wave_target[w];
      FT_CUDA(h, cudaMalloc(&cp.d_wave_target, cp.wave_target.size() * sizeof(int)));
      FT_CUDA(h, cudaMemcpyAsync(cp.d_wave_target, cp.wave_target.data(), cp.wave_target.size() * sizeof(int), cudaMemcpyHostToDevice, stream));
    }
    cp.uploaded = true;
  }
  const int units = cp.plan.units;
  if (enc_front) {
    const int inc = units * CG * (kThreads / 32);
    if (h->d_enc_done == nullptr) {
      FT_CUDA(h, cudaMalloc(&h->d_enc_done, sizeof(int)));
      FT_CUDA(h, cudaMemsetAsync(h->d_enc_done, 0, sizeof(int), stream));
      h->enc_done_value = 0;
    } else if (h->enc_done_value > (1 << 30) - inc) {
      FT_CUDA(h, cudaMemsetAsync(h->d_enc_done, 0, sizeof(int), stream));
      h->enc_done_value = 0;
    }
    h->enc_done_value += inc;
    p.enc_done = h->d_enc_done;
    p.enc_target = h->enc_done_value;
  }
  p.plan = cp.d_items;
  p.plan_off = cp.d_off;
  p.sk_tiles = cp.plan.sk_tiles;
  p.sk_slices = cp.plan.sk_slices;
  if (p.sk_tiles > 0) {
    const size_t flag_bytes = 65536;  // fixed location at the start of the buffer
    const size_t ws_floats = static_cast<size_t>(p.sk_tiles) * (p.sk_slices - 1) * CG * kBM * BN;
    const float *before = h->d_sk;
    rc = ensure_buf(h, &h->d_sk, &h->sk_bytes, flag_bytes + ws_floats * sizeof(float));
    if (rc) return rc;
    p.sk_flags = reinterpret_cast<int *>(h->d_sk);
    p.sk_ws = h->d_sk + flag_bytes / sizeof(float);
    if (h->d_sk != before || h->sk_epoch > (1 << 30)) {  // fresh buffer (or epoch wrap): no flag may alias a live epoch
      FT_CUDA(h, cudaMemsetAsync(p.sk_flags, 0, flag_bytes, stream));
      h->sk_epoch = 0;
    }
    p.sk_epoch = ++h->sk_epoch;
  }
  {
    // Helper-assisted final epilogues (the helper warp of each TMEM lane quadrant takes the upper half of the columns).
    // Measured (profiles/r01_probe24_*, beta = -1.5): ABFT +2.4 % at 1024^3, +5 % at 2048^3, +2 % at 3072^3, +0.8 % at
    // 4096^3, +0.5 % at 8192^3; plain kernel +10.6 % at 1024^3 (one wave: the whole epilogue is exposed), neutral in
    // between, -0.7 % at 8192^3 (the pair barriers cost more than the 3.6 us tail they shorten) -- hence the rule.
    const long long ea = dbg("epi_assist", -2);
    p.epi_assist = ea >= 0 ? (ea != 0) : (ft || cp.plan.items.size() <= 3 * static_cast<size_t>(units));
  }
  {
    // Wave re-synchronisation for problems that run many waves over operands that do not fit L2.  Measured
    // (profiles/r01_probe21_*, r01_trace_16384_per_wave.txt): without it the units' start times drift apart by ~2 us per
    // wave and the tile time grows from 178 to 209 us over the 56 waves of 16384^3; with it the spread stays below 6 us:
    // 16384^3 plain 750 -> 811 TFLOP/s (cuBLAS-TF32 831), ABFT 571-695 -> 721-821; 14336^3 +2-7 % / +3-12 %; neutral
    // between 6144 and 12288, -2 % at 4096 (3 waves) -- hence the wave-count limit.
    const long long ws = dbg("wave_sync", -2);
    const bool on = ws >= 0 ? (ws != 0) : (pin.lockstep && static_cast<int>(cp.wave_target.size()) >= 24);
    if (on && cp.wave_target.size() > 1) {
      const size_t bytes = cp.wave_target.size() * sizeof(int);
      if (h->d_wave_cnt == nullptr || h->wave_cnt_cap < cp.wave_target.size()) {
        if (h->d_wave_cnt) FT_CUDA(h, cudaFree(h->d_wave_cnt));
        h->d_wave_cnt = nullptr;
        FT_CUDA(h, cudaMalloc(&h->d_wave_cnt, bytes));
        h->wave_cnt_cap = cp.wave_target.size();
      }
      FT_CUDA(h, cudaMemsetAsync(h->d_wave_cnt, 0, bytes, stream));
      p.wave_cnt = h->d_wave_cnt;
      p.wave_target = cp.d_wave_target;
    }
  }
  if (dbg("trace", 0) != 0) {
    const int cap = 64;
    if (h->d_trace == nullptr || h->trace_units < units) {
      if (h->d_trace) FT_CUDA(h, cudaFree(h->d_trace));
      h->d_trace = nullptr;
      FT_CUDA(h, cudaMalloc(&h->d_trace, static_cast<size_t>(units) * cap * 8 * sizeof(unsigned long long)));
      h->trace_units = units;
    }
    FT_CUDA(h, cudaMemsetAsync(h->d_trace, 0, static_cast<size_t>(units) * cap * 8 * sizeof(unsigned long long), stream));
    p.trace = h->d_trace;
    p.trace_cap = cap;
  }
  // Programmatic dependent launch by default: the kernel's launch latency and prologue overlap the tail of whatever
  // precedes it in the stream; unless it follows its own pre-pass (pdl_wait = 1: only the checksum items wait) every
  // thread executes griddepcontrol.wait before the first global access.
  if (p.pdl_wait == 0 && dbg("pdl_chain", 1) != 0) p.pdl_wait = 2;
  h->last_stream = stream;
  ++h->launch_count;
  int lrc = FTSGEMM_ERR_UNSUPPORTED;
#define FT_DISPATCH(bn, cg)                                                          \
  if (BN == bn && CG == cg)                                                          \
    lrc = !ft ? launch_tc<bn, false, cg>(h, tmA, tmB, tmC, p, units, stream)         \
              : (o.protect_epilogue ? launch_tc<bn, true, cg, true>(h, tmA, tmB, tmC, p, units, stream) \
                                    : launch_tc<bn, true, cg>(h, tmA, tmB, tmC, p, units, stream));
  FT_DISPATCH(32, 1)
  FT_DISPATCH(64, 1)
  FT_DISPATCH(128, 1)
  FT_DISPATCH(256, 1)
  FT_DISPATCH(64, 2)
  FT_DISPATCH(128, 2)
  FT_DISPATCH(256, 2)
#undef FT_DISPATCH
  return lrc;
}

int run_cublas(ftsgemm_handle_t h, bool tf32, int M, int N, int K, const float *dA, const float *dB, float *dC,
               float alpha, float beta, cudaStream_t stream) {
  FT_CUBLAS(h, cublasSetStream(h->cublas, stream));
  FT_CUBLAS(h, cublasSetPointerMode(h->cublas, CUBLAS_POINTER_MODE_HOST));
  FT_CUBLAS(h, cublasSetMathMode(h->cublas, tf32 ? CUBLAS_TF32_TENSOR_OP_MATH : CUBLAS_DEFAULT_MATH));
  // NT on column-major buffers, as the reference's verification call (sgemm.cu:108)
  FT_CUBLAS(h, cublasSgemm(h->cublas, CUBLAS_OP_N, CUBLAS_OP_T, M, N, K, &alpha, dA, M, dB, N, &beta, dC, M));
  h->last_stream = stream;
  return FTSGEMM_OK;
}

__global__ void fill_kernel(float *p, float v, size_t n) {
  size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  if (i < n) p[i] = v;
}

// 3xTF32: lo = x - tf32(x) (exact in FP32; the tensor core truncates lo to its own 11 significant bits when it reads it)
__global__ void split_lo_kernel(const float4 *__restrict__ x, float4 *__restrict__ lo, size_t n4) {
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n4; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const float4 v = __ldg(x + i);
    float4 r;
    r.x = v.x - __uint_as_float(__float_as_uint(v.x) & 0xFFFFE000u);
    r.y = v.y - __uint_as_float(__float_as_uint(v.y) & 0xFFFFE000u);
    r.z = v.z - __uint_as_float(__float_as_uint(v.z) & 0xFFFFE000u);
    r.w = v.w - __uint_as_float(__float_as_uint(v.w) & 0xFFFFE000u);
    lo[i] = r;
  }
}

// fault verdict of the launches since the last ftsgemm_get_stats, as 8 doubles in device memory (ftsgemm_stats_device)
__global__ void stats_vector_kernel(const DeviceStats *st, double *out) {
  ptx::pdl_wait();  // launched as a programmatic dependent: the GEMM in front of it must have completed
  ptx::pdl_launch_dependents();
  if (threadIdx.x == 0) {
    out[0] = static_cast<double>(st->tiles);
    out[1] = static_cast<double>(st->rows_checked);
    out[2] = static_cast<double>(st->detected);
    out[3] = static_cast<double>(st->corrected);
    out[4] = static_cast<double>(st->uncorrectable);
    out[5] = static_cast<double>(st->checksum_faults);
    out[6] = static_cast<double>(__uint_as_float(st->max_abs_bits));
    out[7] = static_cast<double>(__uint_as_float(st->max_rel_bits));
  }
}

// verify_matrix (utils/utils.cu:61-77) on the device: smallest failing index + Frobenius sums
__global__ void verify_kernel(const float *ref, const float *x, size_t n, unsigned long long *first_bad, double *num,
                              double *den, unsigned long long *bad_count) {
  double ln = 0.0, ld = 0.0;
  unsigned long long lb = ~0ull, nbad = 0;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const double r = ref[i], d = fabs(r - static_cast<double>(x[i]));
    if (((d / fabs(r)) > 0.01 && d > 0.01) || !(d == d)) {
      lb = lb < i ? lb : i;
      ++nbad;
    }
    ln += d * d;
    ld += r * r;
  }
  for (int o = 16; o > 0; o >>= 1) {
    ln += __shfl_xor_sync(0xffffffffu, ln, o);
    ld += __shfl_xor_sync(0xffffffffu, ld, o);
    unsigned long long ob = __shfl_xor_sync(0xffffffffu, lb, o);
    lb = lb < ob ? lb : ob;
    nbad += __shfl_xor_sync(0xffffffffu, nbad, o);
  }
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(num, ln);
    atomicAdd(den, ld);
    atomicMin(first_bad, lb);
    if (nbad) atomicAdd(bad_count, nbad);
  }
}

}  // namespace

// =============================================================================================== C ABI
extern "C" {

int ftsgemm_abi_version(void) { return FTSGEMM_ABI_VERSION; }

const char *ftsgemm_error_string(int code) {
  switch (code) {
    case FTSGEMM_OK: return "ok";
    case FTSGEMM_ERR_INVALID_ARG: return "invalid argument";
    case FTSGEMM_ERR_UNSUPPORTED: return "unsupported shape or kernel id";
    case FTSGEMM_ERR_CUDA: return "CUDA error (see ftsgemm_last_cuda_error)";
    case FTSGEMM_ERR_NO_DEVICE: return "no sm_100 CUDA device available (libftsgemm has no CPU fallback)";
    case FTSGEMM_ERR_CUBLAS: return "cuBLAS error";
    case FTSGEMM_ERR_VERIFY: return "verification failed";
    case FTSGEMM_ERR_TIMEOUT: return "device-side wait timed out (grid not co-resident or protocol error): the launch's result is undefined";
  }
  return "unknown error";
}

void ftsgemm_default_opts(ftsgemm_opts *o) {
  if (!o) return;
  memset(o, 0, sizeof(*o));
  o->struct_size = sizeof(*o);
  o->selftest_value = 10000.0f;  // ft_sgemm_huge.cuh:51
  o->selftest_row = 17;          // ft_sgemm_huge.cuh:49 (tx_injec)
  o->selftest_col = 0;
  o->baseline_host_sync = 1;
}

int ftsgemm_kernel_table(ftsgemm_kernel_info *out, int cap) {
  if (out)
    for (int i = 0; i < kNumVariants && i < cap; ++i) out[i] = kVariants[i].info;
  return kNumVariants;
}

int ftsgemm_select_kernel(int M, int N, int K, int fault_tolerant) {
  if (M <= 0 || N <= 0 || K <= 0) return FTSGEMM_ERR_INVALID_ARG;
  return select_variant(M, N, fault_tolerant != 0);
}

int ftsgemm_kernel_lookup(int kernel_id, ftsgemm_kernel_info *out) {
  const Variant *v = find_variant(kernel_id);
  if (!v) return FTSGEMM_ERR_INVALID_ARG;
  if (out) *out = v->info;
  return FTSGEMM_OK;
}

// Enumerate the work decomposition of one launch on the HOST (same inline code the device runs): for every work unit,
// in processing order, rows of 9 ints {unit, tile, is_chk, m_blk, n_blk, kb_begin, kb_end, kind, slice}.  Returns the
// number of rows (fills min(cap, rows)); hdr[0..7] = {units, num_tiles, n_chk_tiles, sk_tiles, num_kb, cta_group, sk_slices, chk_slices}.
int ftsgemm_debug_schedule(int kernel_id, int M, int N, int K, int num_sms, int *hdr, int *rows, int cap) {
  const Variant *v = find_variant(kernel_id);
  if (!v || v->info.engine != 1 || M <= 0 || N <= 0 || K <= 0 || num_sms <= 0) return FTSGEMM_ERR_INVALID_ARG;
  if (v->bn == 0) v = find_variant(select_variant(M, N, v->info.fault_tolerant != 0));
  KernelParams p;
  memset(&p, 0, sizeof(p));
  p.M = M; p.N = N; p.K = K;
  plan_tiles(M, N, v->bn, v->cg, v->info.fault_tolerant != 0, &p);
  if (v->info.fault_tolerant) {
    if (M % kAtomMN == 0 && N % kAtomMN == 0 && dbg("tma3d", 1) != 0) p.tma3d = 7;
    p.chk_in_carriers = use_carriers(p, num_sms / v->cg, v->cg) ? 1 : 0;
    p.chk_slices = p.chk_in_carriers ? 1 : choose_chk_slices(p, num_sms / v->cg, K);
  }
  const PlanInput pin = make_plan_input(num_sms / v->cg, v->cg, v->bn, K, p);
  const Plan plan = build_plan(pin);
  if (hdr) {
    hdr[0] = plan.units; hdr[1] = pin.n_chk_tiles + pin.n_data_tiles; hdr[2] = pin.n_chk_tiles; hdr[3] = plan.sk_tiles;
    hdr[4] = pin.num_kb; hdr[5] = v->cg; hdr[6] = plan.sk_slices; hdr[7] = pin.chk_slices;
  }
  int n = 0;
  for (int u = 0; u < plan.units; ++u) {
    for (int i = plan.offsets[u]; i < plan.offsets[u + 1]; ++i) {
      const PlanItem &it = plan.items[i];
      if (rows && n < cap) {
        const TileCoord tc = decode_tile(p, it.tile);
        int *r = rows + 9 * n;
        r[0] = u; r[1] = it.tile; r[2] = tc.is_chk ? 1 : 0; r[3] = tc.m_blk; r[4] = tc.n_blk;
        r[5] = it.kb_begin; r[6] = it.kb_end; r[7] = it.kind; r[8] = it.slice;
      }
      ++n;
    }
  }
  return n;
}

int ftsgemm_debug_trace(ftsgemm_handle_t h, unsigned long long *out, int cap_u64) {
  if (!h || !out) return FTSGEMM_ERR_INVALID_ARG;
  if (!h->d_trace) return 0;
  const int n = h->trace_units * 64 * 8;
  if (cap_u64 < n) return FTSGEMM_ERR_INVALID_ARG;
  FT_CUDA(h, cudaDeviceSynchronize());
  FT_CUDA(h, cudaMemcpy(out, h->d_trace, static_cast<size_t>(n) * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  return h->trace_units;
}

int ftsgemm_debug_set(const char *key, long long value) {
  if (!key) return FTSGEMM_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(g_dbg_mu);
  if (value == -1) g_dbg.erase(key);
  else g_dbg[key] = value;
  return FTSGEMM_OK;
}

int ftsgemm_create(ftsgemm_handle_t *out) {
  if (!out) return FTSGEMM_ERR_INVALID_ARG;
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return FTSGEMM_ERR_NO_DEVICE;
  ftsgemm_handle_t h = new ftsgemm_handle_s();
  cudaDeviceProp prop;
  if (cudaGetDevice(&h->device) != cudaSuccess || cudaGetDeviceProperties(&prop, h->device) != cudaSuccess ||
      prop.major != 10) {
    delete h;
    return FTSGEMM_ERR_NO_DEVICE;
  }
  h->num_sms = prop.multiProcessorCount;
  void *fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn) {
    delete h;
    return FTSGEMM_ERR_CUDA;
  }
  h->encode_tiled = reinterpret_cast<EncodeTiledFn>(fn);
  if (cublasCreate(&h->cublas) != CUBLAS_STATUS_SUCCESS) {
    delete h;
    return FTSGEMM_ERR_CUBLAS;
  }
  if (cudaMalloc(&h->d_stats, sizeof(DeviceStats)) != cudaSuccess ||
      cudaMemset(h->d_stats, 0, sizeof(DeviceStats)) != cudaSuccess ||
      cudaMalloc(&h->d_verify, 4 * sizeof(double)) != cudaSuccess) {
    ftsgemm_destroy(h);
    return FTSGEMM_ERR_CUDA;
  }
  *out = h;
  return FTSGEMM_OK;
}

int ftsgemm_destroy(ftsgemm_handle_t h) {
  if (!h) return FTSGEMM_OK;
  DeviceGuard guard(h);
  cudaDeviceSynchronize();
  if (h->cublas) cublasDestroy(h->cublas);
  cudaFree(h->d_stats);
  cudaFree(h->d_chk);
  cudaFree(h->d_chk_out);
  cudaFree(h->d_sk);
  cudaFree(h->d_trace);
  cudaFree(h->d_wave_cnt);
  for (auto &kv : h->plans) {
    cudaFree(kv.second.d_items);
    cudaFree(kv.second.d_off);
    cudaFree(kv.second.d_wave_target);
  }
  cudaFree(h->d_aux);
  cudaFree(h->d_lo);
  cudaFree(h->d_enc_done);
  for (int r = 0; r < kMaxPeers; ++r)
    if (h->peer_opened[r]) cudaIpcCloseMemHandle(h->peer_box[r]);
  cudaFree(h->d_mailbox);
  cudaFree(h->d_exit_count);
  cudaFree(h->d_verify);
  for (int i = 0; i < 3; ++i) cudaFree(h->d_stage[i]);
  if (h->s_in) {
    cudaStreamDestroy(h->s_in);
    cudaStreamDestroy(h->s_out);
    for (int i = 0; i < 16; ++i) {
      cudaEventDestroy(h->ev_in[i]);
      cudaEventDestroy(h->ev_done[i]);
    }
  }
  delete h;
  return FTSGEMM_OK;
}

int ftsgemm_last_cuda_error(ftsgemm_handle_t h) { return h ? h->last_cuda_error : 0; }

unsigned long long ftsgemm_launch_count(ftsgemm_handle_t h) { return h ? h->launch_count : 0ull; }

// Copies the caller's options over the defaults.  struct_size is the caller's sizeof(ftsgemm_opts): anything smaller
// than the first published layout (e.g. 0 from a zero-initialised struct) is an error, not "all defaults".
static int load_opts(const ftsgemm_opts *opts, ftsgemm_opts *o) {
  ftsgemm_default_opts(o);
  if (!opts) return FTSGEMM_OK;
  if (opts->struct_size < FTSGEMM_OPTS_V1_SIZE) return FTSGEMM_ERR_INVALID_ARG;
  memcpy(o, opts, opts->struct_size < sizeof(*o) ? opts->struct_size : sizeof(*o));
  o->struct_size = sizeof(*o);
  if (o->check_segments < 0 || o->check_segments > 4096 || o->precision < 0 || o->precision > 1 || o->inject_mode < 0 || o->inject_mode > 2 || o->protect_epilogue < 0 || o->protect_epilogue > 1 || o->selftest_row < 0 || o->selftest_col < 0 || o->n_faults < 0 ||
      o->n_faults > FTSGEMM_MAX_FAULTS)
    return FTSGEMM_ERR_INVALID_ARG;
  return FTSGEMM_OK;
}

int ftsgemm_run(ftsgemm_handle_t h, int kernel_id, int M, int N, int K, const float *dA, const float *dB, float *dC,
                float alpha, float beta, const ftsgemm_opts *opts) {
  if (!h) return FTSGEMM_ERR_NO_DEVICE;
  if (!dA || !dB || !dC || M <= 0 || N <= 0 || K <= 0) return FTSGEMM_ERR_INVALID_ARG;
  const Variant *v = find_variant(kernel_id);
  if (!v) return FTSGEMM_ERR_INVALID_ARG;
  ftsgemm_opts o;
  const int orc = load_opts(opts, &o);
  if (orc) return orc;
  DeviceGuard guard(h);
  cudaStream_t stream = static_cast<cudaStream_t>(o.stream);
  if (v->info.engine == 1 && v->bn == 0) {  // ids 20 / 40: per-shape choice
    v = find_variant(select_variant(M, N, v->info.fault_tolerant != 0));
    if (!v) return FTSGEMM_ERR_UNSUPPORTED;
  }
  if (v->info.engine == 1 && o.check_segments > 1 && v->info.fault_tolerant) {
    // Intra-K checking (ftsgemm_opts::check_segments): S consecutive K-segments, each a complete fault-tolerant GEMM.  A and
    // B are column-major with k the slow index, so a segment is a pointer offset; segment boundaries are multiples of the
    // stage depth (32 k-rows).  Injected faults (tests) go to the first segment only.
    int S = o.check_segments;
    const int num_kb = (K + kBK - 1) / kBK;
    if (S > num_kb) S = num_kb;
    ftsgemm_opts os = o;
    os.check_segments = 1;
    os.reuse_b_checksums = 0;
    int rc = FTSGEMM_OK;
    for (int sg = 0; sg < S && !rc; ++sg) {
      const int k0 = static_cast<int>(static_cast<long long>(num_kb) * sg / S) * kBK;
      int k1 = static_cast<int>(static_cast<long long>(num_kb) * (sg + 1) / S) * kBK;
      if (k1 > K) k1 = K;
      if (sg > 0) os.inject_mode = 0;
      rc = ftsgemm_run(h, v->info.id, M, N, k1 - k0, dA + static_cast<size_t>(k0) * M, dB + static_cast<size_t>(k0) * N, dC, alpha,
                       sg == 0 ? beta : 1.0f, &os);
    }
    return rc;
  }
  if (v->info.engine == 1 && o.precision == 1) {
    // 3xTF32 (FP32-grade accuracy, the reference's kernels are true FP32 FFMA, ft_sgemm_huge.cuh:228-323): with
    // x = hi + lo (hi = the 11 significant bits the tensor core reads, lo = x - hi exactly),
    //   A B^T ~= A_lo B_hi^T + A_hi B_lo^T + A_hi B_hi^T       (A_lo B_lo^T ~ 2^-22 relative is dropped)
    // as three launches of the same kernel, smallest terms first, each accumulating into C -- every one of them a
    // complete fault-tolerant GEMM with its own checksum vectors, so ABFT covers the whole 3-pass product.
    if ((static_cast<size_t>(M) * K) % 4 || (static_cast<size_t>(N) * K) % 4) return FTSGEMM_ERR_UNSUPPORTED;
    const size_t need = (static_cast<size_t>(M) + N) * K * sizeof(float);
    int rc = ensure_buf(h, &h->d_lo, &h->lo_bytes, need);
    if (rc) return rc;
    float *dAlo = h->d_lo, *dBlo = h->d_lo + static_cast<size_t>(M) * K;
    split_lo_kernel<<<h->num_sms * 8, 256, 0, stream>>>(reinterpret_cast<const float4 *>(dA), reinterpret_cast<float4 *>(dAlo),
                                                        static_cast<size_t>(M) * K / 4);
    split_lo_kernel<<<h->num_sms * 8, 256, 0, stream>>>(reinterpret_cast<const float4 *>(dB), reinterpret_cast<float4 *>(dBlo),
                                                        static_cast<size_t>(N) * K / 4);
    FT_CUDA(h, cudaGetLastError());
    h->launch_count += 2;
    ftsgemm_opts o3 = o;
    o3.reuse_b_checksums = 0;
    o3.precision = 0;
    ftsgemm_opts o_quiet = o3;  // injected faults belong to the main product only
    o_quiet.inject_mode = 0;
    rc = run_tc(h, *v, M, N, K, dAlo, dB, dC, alpha, beta, o_quiet, stream);
    if (!rc) rc = run_tc(h, *v, M, N, K, dA, dBlo, dC, alpha, 1.0f, o_quiet, stream);
    if (!rc) rc = run_tc(h, *v, M, N, K, dA, dB, dC, alpha, 1.0f, o3, stream);
    return rc;
  }
  switch (v->info.engine) {
    case 0: return run_cublas(h, v->info.id == 7, M, N, K, dA, dB, dC, alpha, beta, stream);
    case 1: return run_tc(h, *v, M, N, K, dA, dB, dC, alpha, beta, o, stream);
    case 2: return ftsgemm_baseline(h, M, N, K, dA, dB, dC, alpha, beta, v->info.id == 30 ? 1 : 0, &o, nullptr);
  }
  return FTSGEMM_ERR_UNSUPPORTED;
}

int ftsgemm_get_stats(ftsgemm_handle_t h, ftsgemm_stats *out) {
  if (!h) return FTSGEMM_ERR_NO_DEVICE;
  if (!out) return FTSGEMM_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  FT_CUDA(h, cudaStreamSynchronize(h->last_stream));
  const int arc = check_abort_flag(h);
  if (arc) return arc;
  DeviceStats ds;
  FT_CUDA(h, cudaMemcpy(&ds, h->d_stats, sizeof(ds), cudaMemcpyDeviceToHost));
  FT_CUDA(h, cudaMemset(h->d_stats, 0, sizeof(DeviceStats)));
  memset(out, 0, sizeof(*out));
  out->tiles = ds.tiles;
  out->rows_checked = ds.rows_checked;
  out->detected = ds.detected;
  out->corrected = ds.corrected;
  out->uncorrectable = ds.uncorrectable;
  out->checksum_faults = ds.checksum_faults;
  out->recomputed = ds.recomputed;
  out->epilogue_faults = ds.epilogue_faults;
  memcpy(&out->max_abs_residual, &ds.max_abs_bits, 4);
  memcpy(&out->max_rel_residual, &ds.max_rel_bits, 4);
  out->n_events = ds.n_events < FTSGEMM_MAX_EVENTS ? ds.n_events : FTSGEMM_MAX_EVENTS;
  for (int i = 0; i < out->n_events; ++i) {
    out->events[i].row = ds.events[i].row;
    out->events[i].col = ds.events[i].col;
    out->events[i].residual = ds.events[i].residual;
    out->events[i].corrected_value = ds.events[i].corrected_value;
    out->events[i].status = ds.events[i].status;
  }
  return FTSGEMM_OK;
}

int ftsgemm_peer_export(ftsgemm_handle_t h, void *ipc_handle_64) {
  if (!h) return FTSGEMM_ERR_NO_DEVICE;
  if (!ipc_handle_64) return FTSGEMM_ERR_INVALID_ARG;
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  DeviceGuard guard(h);
  if (!h->d_mailbox) {
    const size_t bytes = static_cast<size_t>(kMaxPeers) * kPeerSlotDoubles * sizeof(double);
    FT_CUDA(h, cudaMalloc(&h->d_mailbox, bytes));
    FT_CUDA(h, cudaMemset(h->d_mailbox, 0, bytes));
    FT_CUDA(h, cudaMalloc(&h->d_exit_count, sizeof(unsigned int)));
    FT_CUDA(h, cudaMemset(h->d_exit_count, 0, sizeof(unsigned int)));
  }
  cudaIpcMemHandle_t hd;
  FT_CUDA(h, cudaIpcGetMemHandle(&hd, h->d_mailbox));
  memcpy(ipc_handle_64, &hd, sizeof(hd));
  return FTSGEMM_OK;
}

int ftsgemm_peer_connect(ftsgemm_handle_t h, int rank, int world, const void *ipc_handles) {
  if (!h) return FTSGEMM_ERR_NO_DEVICE;
  if (!ipc_handles || world < 1 || world > kMaxPeers || rank < 0 || rank >= world || !h->d_mailbox) return FTSGEMM_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  for (int r = 0; r < world; ++r) {
    if (r == rank) {
      h->peer_box[r] = h->d_mailbox;
      continue;
    }
    cudaIpcMemHandle_t hd;
    memcpy(&hd, static_cast<const char *>(ipc_handles) + static_cast<size_t>(r) * sizeof(hd), sizeof(hd));
    void *ptr = nullptr;
    FT_CUDA(h, cudaIpcOpenMemHandle(&ptr, hd, cudaIpcMemLazyEnablePeerAccess));
    h->peer_box[r] = static_cast<double *>(ptr);
    h->peer_opened[r] = true;
  }
  h->peer_rank = rank;
  h->peer_world = world;
  h->peer_seq = 0;
  return FTSGEMM_OK;
}

int ftsgemm_peer_verdict(ftsgemm_handle_t h, double *out8, double *per_rank /* world x 8, may be NULL */, int timeout_ms) {
  if (!h) return FTSGEMM_ERR_NO_DEVICE;
  if (!out8 || h->peer_world < 1) return FTSGEMM_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  FT_CUDA(h, cudaStreamSynchronize(h->last_stream));
  const int arc = check_abort_flag(h);
  if (arc) return arc;
  // every rank's slot must carry (at least) the sequence number of this rank's last publishing launch: the ranks of a
  // tile-sharded product launch the same number of GEMMs
  double box[kMaxPeers * kPeerSlotDoubles];
  const double want = static_cast<double>(h->peer_seq);
  for (int waited = 0;; ++waited) {
    FT_CUDA(h, cudaMemcpy(box, h->d_mailbox, sizeof(double) * h->peer_world * kPeerSlotDoubles, cudaMemcpyDeviceToHost));
    if (timeout_ms < 0) break;  // the caller has synchronised the ranks itself (e.g. a barrier after a stream sync)
    bool all = true;
    for (int r = 0; r < h->peer_world; ++r)
      for (int i = 0; i < 8; ++i) all = all && box[r * kPeerSlotDoubles + 2 * i + 1] >= want;  // (value, sequence) pairs
    if (all) break;
    if (waited >= (timeout_ms > 0 ? timeout_ms : 10000)) return FTSGEMM_ERR_TIMEOUT;
    struct timespec ts = {0, 1000000};
    nanosleep(&ts, nullptr);
  }
  for (int i = 0; i < 8; ++i) out8[i] = 0.0;
  for (int r = 0; r < h->peer_world; ++r) {
    const double *v = box + r * kPeerSlotDoubles;
    for (int i = 0; i < 6; ++i) out8[i] += v[2 * i];
    for (int i = 6; i < 8; ++i) out8[i] = v[2 * i] > out8[i] ? v[2 * i] : out8[i];
    if (per_rank)
      for (int i = 0; i < 8; ++i) per_rank[r * 8 + i] = v[2 * i];
  }
  return FTSGEMM_OK;
}

int ftsgemm_stats_device(ftsgemm_handle_t h, double *d_out8, void *stream_v) {
  if (!h) return FTSGEMM_ERR_NO_DEVICE;
  if (!d_out8) return FTSGEMM_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  // a programmatic dependent of the GEMM it reports on, and a programmatic primary of the next launch: the launch chain
  // of back-to-back steps is not broken by the snapshot
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(1);
  cfg.blockDim = dim3(32);
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = dbg("pdl_chain", 1) != 0 ? 1 : 0;
  const DeviceStats *st = h->d_stats;
  FT_CUDA(h, cudaLaunchKernelEx(&cfg, stats_vector_kernel, st, d_out8));
  ++h->launch_count;
  return FTSGEMM_OK;
}

int ftsgemm_run_host(ftsgemm_handle_t h, int kernel_id, int M, int N, int K, const float *hA, const float *hB,
                     float *hC, float alpha, float beta, const ftsgemm_opts *opts) {
  if (!h) return FTSGEMM_ERR_NO_DEVICE;
  if (!hA || !hB || !hC || M <= 0 || N <= 0 || K <= 0) return FTSGEMM_ERR_INVALID_ARG;
  ftsgemm_opts o;
  const int orc = load_opts(opts, &o);
  if (orc) return orc;
  DeviceGuard guard(h);
  const size_t bytes[3] = {sizeof(float) * M * static_cast<size_t>(K), sizeof(float) * N * static_cast<size_t>(K),
                           sizeof(float) * M * static_cast<size_t>(N)};
  for (int i = 0; i < 3; ++i)
    if (h->stage_bytes[i] < bytes[i]) {
      if (h->d_stage[i]) FT_CUDA(h, cudaFree(h->d_stage[i]));
      h->d_stage[i] = nullptr;
      h->stage_bytes[i] = 0;
      FT_CUDA(h, cudaMalloc(&h->d_stage[i], bytes[i]));
      h->stage_bytes[i] = bytes[i];
    }
  cudaStream_t stream = static_cast<cudaStream_t>(o.stream);
  // Column panels of C pipeline the three phases (the PCIe link is full duplex and the GEMM of a panel takes a few per
  // cent of its transfer time): upload stream  A, B_0, C_0, B_1, C_1, ...;  compute stream  GEMM_j after (A, B_j, C_j);
  // download stream  C_j after GEMM_j.  Panel widths are multiples of the widest tile (256), so every element is
  // accumulated exactly as in the one-shot device path (bit-identical, tests/test_gpu_parity.py).  B_j is a row block of
  // the N x K column-major operand: a 2-D copy into a compact (ld = N_j) staging panel.
  const int max_panels = static_cast<int>(sizeof(h->ev_in) / sizeof(h->ev_in[0]));
  int panels = static_cast<int>(dbg("host_panels", 0));
  if (panels <= 0) panels = N >= 4096 ? 4 : (N >= 2048 ? 2 : 1);
  if (panels > max_panels) panels = max_panels;
  int pw = ((N + panels - 1) / panels + 255) / 256 * 256;  // panel width
  if (pw >= N) {
    pw = N;
    panels = 1;
  } else {
    panels = (N + pw - 1) / pw;
  }
  if (!h->s_in) {
    FT_CUDA(h, cudaStreamCreateWithFlags(&h->s_in, cudaStreamNonBlocking));
    FT_CUDA(h, cudaStreamCreateWithFlags(&h->s_out, cudaStreamNonBlocking));
    for (int i = 0; i < max_panels; ++i) {
      FT_CUDA(h, cudaEventCreateWithFlags(&h->ev_in[i], cudaEventDisableTiming));
      FT_CUDA(h, cudaEventCreateWithFlags(&h->ev_done[i], cudaEventDisableTiming));
    }
  }
  float *dA = h->d_stage[0], *dBs = h->d_stage[1], *dC = h->d_stage[2];
  FT_CUDA(h, cudaMemcpyAsync(dA, hA, bytes[0], cudaMemcpyHostToDevice, h->s_in));
  for (int j = 0; j < panels; ++j) {
    const int n0 = j * pw, nj = (N - n0) < pw ? (N - n0) : pw;
    float *dBj = dBs + static_cast<size_t>(n0) * K;
    if (panels == 1)
      FT_CUDA(h, cudaMemcpyAsync(dBj, hB, bytes[1], cudaMemcpyHostToDevice, h->s_in));
    else
      FT_CUDA(h, cudaMemcpy2DAsync(dBj, sizeof(float) * nj, hB + n0, sizeof(float) * N, sizeof(float) * nj, K,
                                   cudaMemcpyHostToDevice, h->s_in));
    if (beta != 0.0f)
      FT_CUDA(h, cudaMemcpyAsync(dC + static_cast<size_t>(n0) * M, hC + static_cast<size_t>(n0) * M,
                                 sizeof(float) * M * static_cast<size_t>(nj), cudaMemcpyHostToDevice, h->s_in));
    FT_CUDA(h, cudaEventRecord(h->ev_in[j], h->s_in));
  }
  o.reuse_b_checksums = 0;  // the staging buffer content changed
  for (int j = 0; j < panels; ++j) {
    const int n0 = j * pw, nj = (N - n0) < pw ? (N - n0) : pw;
    FT_CUDA(h, cudaStreamWaitEvent(stream, h->ev_in[j], 0));
    const int rc = ftsgemm_run(h, kernel_id, M, nj, K, dA, dBs + static_cast<size_t>(n0) * K, dC + static_cast<size_t>(n0) * M,
                               alpha, beta, &o);
    if (rc) {
      cudaStreamSynchronize(h->s_in);
      cudaStreamSynchronize(h->s_out);
      return rc;
    }
    FT_CUDA(h, cudaEventRecord(h->ev_done[j], stream));
    FT_CUDA(h, cudaStreamWaitEvent(h->s_out, h->ev_done[j], 0));
    FT_CUDA(h, cudaMemcpyAsync(hC + static_cast<size_t>(n0) * M, dC + static_cast<size_t>(n0) * M,
                               sizeof(float) * M * static_cast<size_t>(nj), cudaMemcpyDeviceToHost, h->s_out));
  }
  FT_CUDA(h, cudaStreamSynchronize(h->s_out));
  FT_CUDA(h, cudaStreamSynchronize(stream));
  return check_abort_flag(h);
}

int ftsgemm_baseline(ftsgemm_handle_t h, int M, int N, int K, const float *dA, const float *dB, float *dC,
                     float alpha, float beta, int math_mode, const ftsgemm_opts *opts, float *residual_out) {
  if (!h) return FTSGEMM_ERR_NO_DEVICE;
  if (!dA || !dB || !dC || M <= 0 || N <= 0 || K <= 0) return FTSGEMM_ERR_INVALID_ARG;
  ftsgemm_opts o;
  const int orc = load_opts(opts, &o);
  if (orc) return orc;
  DeviceGuard guard(h);
  cudaStream_t stream = static_cast<cudaStream_t>(o.stream);
  const bool host_sync = o.baseline_host_sync != 0;
  const int mx = M > N ? M : N;
  // aux layout: ones[mx] | c_row[M] | c_col[N] | a_col[256] | b_row[256] | acol_x_b[N] | brow_x_a[M] | res[2] | consts[3]
  const size_t need = static_cast<size_t>(mx) + M + N + 256 + 256 + N + M + 2 + 3;
  if (h->aux_floats < need) {
    if (h->d_aux) FT_CUDA(h, cudaFree(h->d_aux));
    h->d_aux = nullptr;
    h->aux_floats = 0;
    FT_CUDA(h, cudaMalloc(&h->d_aux, need * sizeof(float)));
    h->aux_floats = need;
  }
  float *ones = h->d_aux, *c_row = ones + mx, *c_col = c_row + M, *a_col = c_col + N, *b_row = a_col + 256,
        *acol_x_b = b_row + 256, *brow_x_a = acol_x_b + N, *res = brow_x_a + M;
  fill_kernel<<<(mx + 255) / 256, 256, 0, stream>>>(ones, 1.0f, mx);
  FT_CUDA(h, cudaGetLastError());
  FT_CUBLAS(h, cublasSetStream(h->cublas, stream));
  FT_CUBLAS(h, cublasSetMathMode(h->cublas, math_mode ? CUBLAS_TF32_TENSOR_OP_MATH : CUBLAS_DEFAULT_MATH));
  const float one = 1.0f, zero = 0.0f, neg1 = -1.0f;
  for (int k0 = 0; k0 < K; k0 += 256) {
    const int kc = (K - k0) < 256 ? (K - k0) : 256;
    const float beta_eff = (k0 == 0) ? beta : 1.0f;
    const float *Ac = dA + static_cast<size_t>(k0) * M;
    const float *Bc = dB + static_cast<size_t>(k0) * N;
    FT_CUBLAS(h, cublasSetPointerMode(h->cublas, CUBLAS_POINTER_MODE_HOST));
    // product chunk (baseline_ft_sgemm.cuh:6)
    FT_CUBLAS(h, cublasSgemm(h->cublas, CUBLAS_OP_N, CUBLAS_OP_T, M, N, kc, &alpha, Ac, M, Bc, N, &beta_eff, dC, M));
    if (host_sync) FT_CUDA(h, cudaStreamSynchronize(stream));
    // row / column sums of all of C (:9,:12) -- the re-read of C the fused kernel removes
    FT_CUBLAS(h, cublasSgemv(h->cublas, CUBLAS_OP_N, M, N, &one, dC, M, ones, 1, &zero, c_row, 1));
    FT_CUBLAS(h, cublasSgemv(h->cublas, CUBLAS_OP_T, M, N, &one, dC, M, ones, 1, &zero, c_col, 1));
    // encode: e^T A_chunk (:15) and B_chunk^T e (:18)
    FT_CUBLAS(h, cublasSgemv(h->cublas, CUBLAS_OP_T, M, kc, &one, Ac, M, ones, 1, &zero, a_col, 1));
    FT_CUBLAS(h, cublasSgemv(h->cublas, CUBLAS_OP_T, N, kc, &one, Bc, N, ones, 1, &zero, b_row, 1));
    if (host_sync) FT_CUDA(h, cudaStreamSynchronize(stream));
    // checksum products (:21,:24); accumulated over chunks so that, for alpha = 1 and beta = 0, the residual of
    // the last chunk is the residual of the whole product
    const float *acc_beta = (k0 == 0) ? &zero : &one;
    FT_CUBLAS(h, cublasSgemv(h->cublas, CUBLAS_OP_N, N, kc, &one, Bc, N, a_col, 1, acc_beta, acol_x_b, 1));
    FT_CUBLAS(h, cublasSgemv(h->cublas, CUBLAS_OP_N, M, kc, &one, Ac, M, b_row, 1, acc_beta, brow_x_a, 1));
    if (host_sync) FT_CUDA(h, cudaStreamSynchronize(stream));
    // residual + reduce (:27-31); dot results land in device memory
    FT_CUBLAS(h, cublasSaxpy(h->cublas, N, &neg1, acol_x_b, 1, c_col, 1));
    FT_CUBLAS(h, cublasSetPointerMode(h->cublas, CUBLAS_POINTER_MODE_DEVICE));
    FT_CUBLAS(h, cublasSdot(h->cublas, N, c_col, 1, ones, 1, res));
    if (host_sync) FT_CUDA(h, cudaStreamSynchronize(stream));
    FT_CUBLAS(h, cublasSetPointerMode(h->cublas, CUBLAS_POINTER_MODE_HOST));
    FT_CUBLAS(h, cublasSaxpy(h->cublas, M, &neg1, brow_x_a, 1, c_row, 1));
    FT_CUBLAS(h, cublasSetPointerMode(h->cublas, CUBLAS_POINTER_MODE_DEVICE));
    FT_CUBLAS(h, cublasSdot(h->cublas, M, c_row, 1, ones, 1, res + 1));
  }
  FT_CUBLAS(h, cublasSetPointerMode(h->cublas, CUBLAS_POINTER_MODE_HOST));
  if (residual_out)
    FT_CUDA(h, cudaMemcpyAsync(residual_out, res, 2 * sizeof(float), cudaMemcpyDeviceToDevice, stream));
  h->last_stream = stream;
  return FTSGEMM_OK;
}

int ftsgemm_verify(ftsgemm_handle_t h, const float *d_ref, const float *d_x, int M, int N, long long *first_bad,
                   double *rel_fro, void *stream_v) {
  if (!h) return FTSGEMM_ERR_NO_DEVICE;
  if (!d_ref || !d_x || M <= 0 || N <= 0) return FTSGEMM_ERR_INVALID_ARG;
  DeviceGuard guard(h);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  unsigned long long init[4];
  init[0] = ~0ull;
  double z = 0.0;
  memcpy(&init[1], &z, 8);
  memcpy(&init[2], &z, 8);
  init[3] = 0;
  FT_CUDA(h, cudaMemcpyAsync(h->d_verify, init, sizeof(init), cudaMemcpyHostToDevice, stream));
  const size_t n = static_cast<size_t>(M) * N;
  verify_kernel<<<h->num_sms * 8, 256, 0, stream>>>(d_ref, d_x, n, reinterpret_cast<unsigned long long *>(h->d_verify),
                                                   h->d_verify + 1, h->d_verify + 2,
                                                   reinterpret_cast<unsigned long long *>(h->d_verify + 3));
  FT_CUDA(h, cudaGetLastError());
  unsigned long long res[4];
  FT_CUDA(h, cudaMemcpyAsync(res, h->d_verify, sizeof(res), cudaMemcpyDeviceToHost, stream));
  FT_CUDA(h, cudaStreamSynchronize(stream));
  double num, den;
  memcpy(&num, &res[1], 8);
  memcpy(&den, &res[2], 8);
  if (first_bad) *first_bad = res[0] == ~0ull ? -1 : static_cast<long long>(res[0]);
  if (rel_fro) *rel_fro = den > 0 ? sqrt(num / den) : sqrt(num);
  h->last_verify_bad = res[3];
  return res[0] == ~0ull ? FTSGEMM_OK : FTSGEMM_ERR_VERIFY;
}

long long ftsgemm_verify_bad_count(ftsgemm_handle_t h) { return h ? static_cast<long long>(h->last_verify_bad) : -1; }

}  // extern "C"
