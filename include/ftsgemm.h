/*
 * ftsgemm.h -- C ABI of libftsgemm.so: fused fault-tolerant (ABFT) SGEMM for NVIDIA B200 (sm_100a).
 *
 * This is the drop-in boundary for the ONE hot path of
 * shixun404/Fault-Tolerant-SGEMM-on-NVIDIA-GPUs.  The reference exposes no library API; its boundary is
 *   (1) the process CLI   ft_sgemm START END GAP ST_KERNEL END_KERNEL   (kernel/ft_sgemm/sgemm.cu:13-19),
 *   (2) the uniform kernel contract
 *         void k(int M,int N,int K,float*A,float*B,float*C,float alpha,float beta)
 *       (kernel/ft_sgemm/include_code_gen/ft_sgemm_huge.cuh:11) selected by a kernel id
 *       (dispatch chains sgemm.cu:110-199 / :256-430, id+name tables sgemm.cu:235-237,
 *        tile table code_gen/main.py:8-16),
 *   (3) the non-fused baseline  baseline_ft_sgemm(...)  (kernel/ft_sgemm/include/baseline_ft_sgemm.cuh:1).
 * Every entry point below names the reference interface it replaces.  Plain C types only: device/host
 * pointers, ints, floats; no torch / C++ types.
 *
 * Data layout (identical to the reference kernels): A is M x K column-major (ld = M), B is N x K
 * column-major (ld = N), C is M x N column-major (ld = M);  C = alpha * A * B^T + beta * C  in place.
 * All functions return FTSGEMM_OK (0) or a negative FTSGEMM_ERR_* code; nothing calls exit().
 */
#ifndef FTSGEMM_H_
#define FTSGEMM_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FTSGEMM_ABI_VERSION 2

enum {
  FTSGEMM_OK = 0,
  FTSGEMM_ERR_INVALID_ARG = -1,  /* bad pointer / size / id */
  FTSGEMM_ERR_UNSUPPORTED = -2,  /* shape not supported by the selected variant */
  FTSGEMM_ERR_CUDA = -3,         /* a CUDA runtime/driver call failed; see ftsgemm_last_cuda_error */
  FTSGEMM_ERR_NO_DEVICE = -4,    /* no sm_100 device / driver (the product has NO CPU fallback) */
  FTSGEMM_ERR_CUBLAS = -5,
  FTSGEMM_ERR_VERIFY = -6,       /* used by the driver helpers only */
  FTSGEMM_ERR_TIMEOUT = -7       /* a device-side wait of the persistent kernel timed out (its CTAs were not all resident,
                                    e.g. the SMs were taken by another context): reported by the next synchronising call
                                    (ftsgemm_get_stats, ftsgemm_run_host); the affected launch's output is undefined, the
                                    CUDA context stays usable */
};

/* Kernel ids: the reference's table (sgemm.cu:235-237) is kept verbatim for ids 0,1-6,10,11-16.
 * ids 7-9 fall through to cuBLAS in the reference (sgemm.cu:197-199); here 7 = cuBLAS with TF32 tensor-op math
 * (the "fault-free cuBLAS TF32" bar), 8-9 = cuBLAS FP32.  ids >= 20 are B200-only extras. */
enum {
  FTSGEMM_ID_CUBLAS = 0,
  FTSGEMM_ID_SGEMM_SMALL = 1, FTSGEMM_ID_SGEMM_MEDIUM = 2, FTSGEMM_ID_SGEMM_LARGE = 3,
  FTSGEMM_ID_SGEMM_TALL = 4, FTSGEMM_ID_SGEMM_WIDE = 5, FTSGEMM_ID_SGEMM_HUGE = 6,
  FTSGEMM_ID_CUBLAS_TF32 = 7,
  FTSGEMM_ID_ABFT_BASELINE = 10,
  FTSGEMM_ID_ABFT_SMALL = 11, FTSGEMM_ID_ABFT_MEDIUM = 12, FTSGEMM_ID_ABFT_LARGE = 13,
  FTSGEMM_ID_ABFT_TALL = 14, FTSGEMM_ID_ABFT_WIDE = 15, FTSGEMM_ID_ABFT_HUGE = 16,
  FTSGEMM_ID_SGEMM_AUTO = 20,        /* plain tcgen05 kernel, variant chosen per shape (ftsgemm_select_kernel)  (B200 extra) */
  FTSGEMM_ID_SGEMM_GIANT = 21,       /* 256 x 256 tile on a CTA pair (cta_group::2), plain  (B200 extra) */
  FTSGEMM_ID_SGEMM_PAIR128 = 22,     /* 256 x 128 tile on a CTA pair, plain: alias of "large" (id 3) */
  FTSGEMM_ID_ABFT_BASELINE_TF32 = 30,/* non-fused baseline with TF32 tensor-op math */
  FTSGEMM_ID_ABFT_GIANT = 31,        /* 256 x 256 CTA-pair tile, fused ABFT: the bench configuration (B200 extra) */
  FTSGEMM_ID_ABFT_PAIR128 = 32,      /* 256 x 128 CTA-pair tile, fused ABFT: alias of "large" (id 13) */
  FTSGEMM_ID_ABFT_AUTO = 40          /* fused ABFT, variant chosen per shape (ftsgemm_select_kernel)  (B200 extra) */
};

typedef struct ftsgemm_handle_s *ftsgemm_handle_t;

/* One row of the kernel-variant table (replaces the id/name arrays at sgemm.cu:235-237 and the
 * tile table at code_gen/main.py:8-16). */
typedef struct ftsgemm_kernel_info {
  int id;
  char name[24];         /* reference row label, e.g. "abft_kernel_huge" */
  int fault_tolerant;    /* 1 = online ABFT fused into the kernel */
  int engine;            /* 0 = cuBLAS, 1 = tcgen05 fused kernel, 2 = cuBLAS call sequence (baseline) */
  int ref_tile_m, ref_tile_n, ref_tile_k; /* the reference's CUDA-core CTA tile (0 for library rows) */
  int tile_m, tile_n, tile_k;             /* this build's sm_100a CTA tile (UMMA M x N, K per smem stage) */
} ftsgemm_kernel_info;

/* Fault to inject into the FP32 accumulator tile in tensor memory, before the checksum test
 * (generalises the reference's always-on injector, ft_sgemm_huge.cuh:49-51,324-327). */
typedef struct ftsgemm_fault {
  int row, col;          /* global element (m, n) of C */
  int mode;              /* 0: acc += add_value      1: acc bits ^= xor_mask (single/multi bit flip)
                          * epilogue upsets (what opts.protect_epilogue detects; the accumulator check has already passed):
                          * 2: acc bits ^= xor_mask in tensor memory AFTER the check, before the store pass re-reads it
                          * 3: the value alpha*acc + beta*c about to be stored has its bits ^= xor_mask (injected by the
                          *    protected store pass only: ignored without opts.protect_epilogue) */
  float add_value;
  uint32_t xor_mask;
} ftsgemm_fault;

#define FTSGEMM_MAX_FAULTS 8
#define FTSGEMM_MAX_EVENTS 16

typedef struct ftsgemm_opts {
  uint32_t struct_size;  /* sizeof(ftsgemm_opts), for ABI evolution */
  void *stream;          /* cudaStream_t; NULL = default stream (the reference uses only the default stream) */
  /* fault injection */
  int inject_mode;       /* 0 none | 1 reference self-test: every CTA tile gets +selftest_value at
                            (selftest_row, selftest_col) of the tile | 2 explicit list faults[0..n_faults) */
  float selftest_value;  /* reference: 10000 */
  int selftest_row, selftest_col;
  int n_faults;
  ftsgemm_fault faults[FTSGEMM_MAX_FAULTS];
  /* detection threshold: a row is flagged when |expected - actual row checksum| > tau_abs + tau_rel * sum_n|acc|.
   * <= 0 selects the calibrated defaults (DESIGN.md section 5): tau_abs = 1e-3, tau_rel = max(1e-5, 1.2e-9 * K), or
   * max(1e-5, 2.5e-8 * K) when the checksum items run as K-slices -- measured fault-free floors of |d1| / sum|acc|: <= 2.3e-6
   * up to 16384^3 on zero-mean operands, ~5.2e-9 * K with non-negative operands and K-slices.  The reference uses the constant 9500
   * (ft_sgemm_huge.cuh:50). */
  float tau_abs, tau_rel;
  int detect_only;       /* 1: count detections but do not correct */
  int reuse_b_checksums; /* 1: B is unchanged since the previous FT call on this handle -> reuse its checksum vectors
                            (no encoder items in this launch) */
  int baseline_host_sync;/* id 10/30: 1 = host-synchronise between stages like the reference
                            (baseline_ft_sgemm.cuh:7,19,26,30); 0 = stream-ordered */
  /* ---- ABI version 2 ---- */
  int precision;         /* 0 (default): single-pass TF32 (operands truncated to 11 significant bits by the tensor core,
                            FP32 accumulate; norm-wise 1e-3 against FP32) | 1: 3xTF32 -- hi/lo split of A and B, three
                            fault-tolerant passes A_lo*B + A*B_lo + A*B: FP32-grade, element-wise parity with the
                            reference's FP32 FFMA kernels (ft_sgemm_huge.cuh:228-323) at ~1/3 of the throughput */
  int check_segments;    /* 0 / 1 (default): one check per tile over the whole K range.  S > 1: intra-K checking -- the product is
                            formed as S consecutive K-segments (S launches, C += alpha * A[:, seg] * B[:, seg]^T), each a
                            complete fault-tolerant GEMM whose tiles are verified and repaired before the segment is
                            committed to C: an upset is caught within K/S of where it happened, and upsets in different
                            segments of one row are each correctable (the reference checks its register accumulators every
                            K/20 iterations, ft_sgemm_huge.cuh:324, code_gen.py:333).  Costs S launches and S passes over C. */
  int no_recompute;      /* 0 (default): a row that is flagged but cannot be repaired from its two checksums (upset too
                            small to locate, two upsets in one row) is RECOMPUTED from A and B on CUDA cores and counted
                            in stats.recomputed -- nothing detected is stored as computed; 1: leave such rows as computed
                            and count them in stats.uncorrectable (round-1 behaviour) */
  int protect_epilogue;  /* 1: the store pass is checked as well (the reference's epilogue c = alpha*res + beta*c,
                            ft_sgemm_huge.cuh:573-690, is unprotected -- and so is the window between the accumulator check
                            and the store): every warp re-sums the accumulator values it re-reads (must equal, bit for bit,
                            the sums the check verified) and sums what it stores (must equal alpha * that + beta * sum of the
                            old values within rounding).  A row segment that fails is counted in stats.epilogue_faults
                            and, when beta == 0, recomputed from A and B; with beta != 0 the old values are gone: it is
                            counted in stats.uncorrectable.  Tiles that are ragged in N are not covered; Inf / NaN already in the old C are
                            not verifiable and not flagged.  A separate kernel instantiation (the default one has no register to
                            spare); measured cost, id 31: +6 % at 8192^3, +18 % at 4096^3, +52 % at 2048^3
                            (profiles/r02_protect_epilogue_cost.jsonl). */
} ftsgemm_opts;
/* sizeof(ftsgemm_opts) of ABI version 1: the smallest struct_size the library accepts (a zero-initialised struct is
 * rejected with FTSGEMM_ERR_INVALID_ARG instead of silently meaning "all defaults on the default stream"). */
#define FTSGEMM_OPTS_V1_SIZE (offsetof(ftsgemm_opts, baseline_host_sync) + sizeof(int))

typedef struct ftsgemm_event {
  int row, col;          /* global element that was located (col = -1 if not locatable) */
  float residual;        /* expected - actual row checksum */
  float corrected_value; /* accumulator value after correction */
  int status;            /* 1 corrected, 2 detected only (detect_only), 3 uncorrectable, 4 checksum-column fault,
                            5 row recomputed, 6 epilogue fault (row segment recomputed), 7 epilogue fault left in C (beta != 0) */
} ftsgemm_event;

typedef struct ftsgemm_stats {
  unsigned long long tiles;        /* CTA tiles processed */
  unsigned long long rows_checked; /* row checksums tested */
  unsigned long long detected;     /* rows whose residual exceeded the threshold */
  unsigned long long corrected;    /* single-element corrections applied */
  unsigned long long uncorrectable;/* detected, not locatable (multi-error row / ambiguous) AND left as computed
                                      (only with opts.no_recompute or detect_only) */
  unsigned long long checksum_faults; /* residual explained by a fault in the checksum column itself */
  float max_abs_residual;          /* max |expected - actual| over all fault-free rows */
  float max_rel_residual;          /* max |expected - actual| / sum_n|acc| over all fault-free rows */
  int n_events;
  ftsgemm_event events[FTSGEMM_MAX_EVENTS];
  /* ---- ABI version 2 ---- */
  unsigned long long recomputed;   /* rows detected but not correctable from the checksums, recomputed on CUDA cores */
  unsigned long long epilogue_faults; /* row segments whose store pass failed its check (opts.protect_epilogue) */
} ftsgemm_stats;

/* ---- lifetime ---------------------------------------------------------------------------------------- */
int ftsgemm_create(ftsgemm_handle_t *out);   /* binds to the current CUDA device; owns cuBLAS handle + workspace.
                                                 A handle is one in-order context: calls on it must be issued from one
                                                 stream at a time (use one handle per concurrently used stream). */
int ftsgemm_destroy(ftsgemm_handle_t h);
int ftsgemm_abi_version(void);
const char *ftsgemm_error_string(int code);
int ftsgemm_last_cuda_error(ftsgemm_handle_t h); /* cudaError_t / CUresult of the last failure, 0 if none */
/* Number of kernels of THIS library (fused GEMM, encode pre-pass, hi/lo split, verdict snapshot; not cuBLAS') launched
 * through the handle since it was created: a fused ABFT GEMM is 1 launch (the encode is a front phase of the kernel),
 * 2 below ~8 MB of B (separate pre-pass) -- what bench.py reports as gpu_launches. */
unsigned long long ftsgemm_launch_count(ftsgemm_handle_t h);
void ftsgemm_default_opts(ftsgemm_opts *o);

/* ---- kernel-variant table  (replaces sgemm.cu:235-237 + code_gen/main.py:8-16) --------------------------- */
int ftsgemm_kernel_table(ftsgemm_kernel_info *out, int cap); /* returns number of rows (fills min(cap, rows)) */
int ftsgemm_kernel_lookup(int kernel_id, ftsgemm_kernel_info *out);
/* The concrete tcgen05 kernel id that ids 20 / 40 (AUTO) resolve to for this shape (replaces the reference's manual
 * choice of a variant per run, sgemm.cu:110-199).  Returns the id (> 0) or a negative error code. */
int ftsgemm_select_kernel(int M, int N, int K, int fault_tolerant);

/* ---- the kernel contract  (replaces `kernel<<<grid,block>>>(M,N,K,dA,dB,dC,alpha,beta)` selected by id,
 *      sgemm.cu:110-199, and cublasSgemm at sgemm.cu:108,198,260) ---------------------------------------------
 * Device pointers, caller-owned, in place on C, asynchronous on opts->stream.  Preconditions as in the
 * reference: 16-byte aligned pointers, M % 4 == 0 and N % 4 == 0 (16-byte rows for TMA); unlike the reference,
 * M/N/K need not be multiples of the tile (TMA zero-fills the ragged edge).  K >= 1. */
int ftsgemm_run(ftsgemm_handle_t h, int kernel_id, int M, int N, int K, const float *dA, const float *dB,
                float *dC, float alpha, float beta, const ftsgemm_opts *opts);

/* Counters of all FT launches since the previous call (synchronises the handle's last stream, then resets). */
int ftsgemm_get_stats(ftsgemm_handle_t h, ftsgemm_stats *out);

/* The same counters as a device-side vector, asynchronously on `stream` and WITHOUT resetting them: d_out8 (device
 * memory, 8 doubles) = {tiles, rows_checked, detected, corrected, uncorrectable, checksum_faults, max_abs_residual,
 * max_rel_residual} of all FT launches since the previous ftsgemm_get_stats.  This is the vector the tile-sharded
 * multi-GPU path exchanges (NCCL all-gather / all-reduce on the same stream) so that every rank agrees on the fault
 * verdict of a distributed product without a host round trip (new work: the reference is single-GPU, sgemm.cu:34). */
int ftsgemm_stats_device(ftsgemm_handle_t h, double *d_out8, void *stream);

/* ---- multi-GPU verdict exchange fused into the GEMM kernel (new work: the reference is single-GPU, sgemm.cu:34) ----------
 * For a product that is tile-sharded over the GPUs of one box (one process per GPU).  Each rank exports the CUDA-IPC handle of
 * its verdict mailbox (ftsgemm_peer_export, 64 bytes), the ranks exchange the handles by any means (the bench uses
 * torch.distributed.all_gather_object), and ftsgemm_peer_connect maps all of them.  From then on the last CTA of every
 * fault-tolerant launch on this handle stores the handle's verdict vector (the 8 doubles of ftsgemm_stats_device), each value
 * paired with the launch's sequence number in one 16-byte store, into slot `rank` of EVERY rank's mailbox -- peer stores over NVLink from inside the GEMM kernel,
 * no collective launch.  ftsgemm_peer_verdict synchronises this handle's stream, waits (up to timeout_ms, default 10 s)
 * until every rank's slot carries the sequence number of this rank's latest launch (the ranks launch the same number of
 * GEMMs), and returns the reduced verdict: counters summed, residual maxima max-ed; per_rank (world x 8 doubles) optional.
 * timeout_ms < 0: no waiting -- for callers that have synchronised the ranks themselves (stream sync + a barrier). */
int ftsgemm_peer_export(ftsgemm_handle_t h, void *ipc_handle_64bytes);
int ftsgemm_peer_connect(ftsgemm_handle_t h, int rank, int world, const void *ipc_handles /* world x 64 bytes */);
int ftsgemm_peer_verdict(ftsgemm_handle_t h, double *out8, double *per_rank, int timeout_ms);

/* Same contract with HOST buffers, synchronous: the call the e2e benchmark times.  The transfers are pipelined over
 * column panels of C (upload A, then per panel B_j (+ C_j when beta != 0) | GEMM_j | download C_j on three streams), so
 * the step costs about the upload time of A, B, C (PCIe is full duplex); pass page-locked host memory for that to
 * hold.  Results are bit-identical to the device path.  Staging buffers / streams are cached on the handle. */
int ftsgemm_run_host(ftsgemm_handle_t h, int kernel_id, int M, int N, int K, const float *hA, const float *hB,
                     float *hC, float alpha, float beta, const ftsgemm_opts *opts);

/* ---- non-fused ABFT baseline  (replaces baseline_ft_sgemm(), include/baseline_ft_sgemm.cuh:1-33) -----------
 * Same call sequence per 256-wide K chunk (1 Sgemm + 6 Sgemv + 2 x (Saxpy + Sdot)), detection only.
 * Differences from the reference, by design: chunks after the first accumulate with beta = 1 so the result is
 * a correct GEMM; Sdot results go to device memory in device-pointer mode; the last chunk may be < 256 wide.
 * math_mode 0 = FP32 (reference), 1 = TF32 tensor-op.  residual_out (device, 2 floats, may be NULL) receives
 * the last chunk's summed column / row residuals. */
int ftsgemm_baseline(ftsgemm_handle_t h, int M, int N, int K, const float *dA, const float *dB, float *dC,
                     float alpha, float beta, int math_mode, const ftsgemm_opts *opts, float *residual_out);

/* ---- comparator (replaces verify_matrix, utils/utils.cu:61-77) on device buffers -------------------------
 * Returns FTSGEMM_OK when every element passes the reference rule (fails iff rel > 1e-2 AND abs > 1e-2),
 * FTSGEMM_ERR_VERIFY otherwise.  first_bad (may be NULL) receives the smallest failing linear index or -1;
 * rel_fro (may be NULL) the Frobenius-norm relative error. */
int ftsgemm_verify(ftsgemm_handle_t h, const float *d_ref, const float *d_x, int M, int N, long long *first_bad,
                   double *rel_fro, void *stream);

/* Number of elements that failed the rule in the last ftsgemm_verify call on this handle (the reference stops at the
 * first; single-pass TF32 legitimately leaves a ~1e-5 fraction of near-zero elements outside 1 %/0.01 for K >= 1024). */
long long ftsgemm_verify_bad_count(ftsgemm_handle_t h);

/* ---- internal / experiments (not part of the drop-in surface) ---------------------------------------------- */
int ftsgemm_debug_set(const char *key, long long value);
/* Host-side enumeration of the work decomposition of one launch (split-K head + data-parallel body), for tests:
 * rows of 9 ints {unit, tile, is_chk, m_blk, n_blk, kb_begin, kb_end, kind(0 whole,1 contributor,2 finisher), slice};
 * hdr[8] = {units, num_tiles, n_chk_tiles, sk_tiles, num_kb, cta_group, sk_slices, chk_slices}; checksum tiles carry
 * their K-slice index in the `slice` column.  Needs no GPU. */
int ftsgemm_debug_schedule(int kernel_id, int M, int N, int K, int num_sms, int *hdr, int *rows, int cap);
/* Device timeline of the last tensor-core launch made with ftsgemm_debug_set("trace", 1): per work unit 64 items x 8
 * u64 = %globaltimer ns {producer start, producer end, MMA start, MMA issue end, accumulator complete, check done,
 * epilogue end, tile | kind << 24}.  Returns the number of units (out must hold units * 512 u64), 0 if none. */
int ftsgemm_debug_trace(ftsgemm_handle_t h, unsigned long long *out, int cap_u64);

#ifdef __cplusplus
}
#endif
#endif /* FTSGEMM_H_ */
