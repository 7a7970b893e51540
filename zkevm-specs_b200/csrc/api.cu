// api.cu — the C-ABI of libzkcheck.so (include/zkcheck.h): context, uploads, lookup-index
// cache, kernel dispatch, result transport.  Unity build: the circuit kernels are included
// below so the whole library is one translation unit (nvcc -gencode arch=compute_100a,
// code=sm_100a).  No torch types cross this boundary.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/zk_constraints.h"
#include "../../include/zkcheck.h"
#include "bytecode.cu"
#include "copy.cu"
#include "evm.cu"
#include "exp.cu"
#include "pi.cu"
#include "assign.cu"
#include "tx.cu"
#include "state.cu"
#include "withdrawal.cu"
#include "circuit.cuh"

using namespace zk;

// ------------------------------------------------------------------ catalogue tables
struct ConstraintInfo {
  const char* name;
  int cls;
  const char* doc;
};
#define ZK_INFO_ENTRY(id, cls, doc) {#id, cls, doc},
static const ConstraintInfo kBytecodeInfo[] = {ZK_BYTECODE_CONSTRAINTS(ZK_INFO_ENTRY)};
static const ConstraintInfo kEvmInfo[] = {ZK_EVM_CONSTRAINTS(ZK_INFO_ENTRY)};
static const ConstraintInfo kCopyInfo[] = {ZK_COPY_CONSTRAINTS(ZK_INFO_ENTRY)};
static const ConstraintInfo kStateInfo[] = {ZK_STATE_CONSTRAINTS(ZK_INFO_ENTRY)};
static const ConstraintInfo kExpInfo[] = {ZK_EXP_CONSTRAINTS(ZK_INFO_ENTRY)};
static const ConstraintInfo kTxInfo[] = {ZK_TX_CONSTRAINTS(ZK_INFO_ENTRY)};
static const ConstraintInfo kSigInfo[] = {ZK_SIG_CONSTRAINTS(ZK_INFO_ENTRY)};
static const ConstraintInfo kPiInfo[] = {ZK_PI_CONSTRAINTS(ZK_INFO_ENTRY)};
static const ConstraintInfo kWdInfo[] = {ZK_WD_CONSTRAINTS(ZK_INFO_ENTRY)};

static const int kCircuitCols[ZK_N_CIRCUITS] = {12, 57, 20, 13, 21, 14, 21, 28, 8};
static const int kTableCols[ZK_N_TABLES] = {4, 6, 14, 5, 4, 14, 5, 12, 2, 4, 3, 11, 3};

static const ConstraintInfo* circuit_info(int circuit, int* n) {
  switch (circuit) {
    case ZK_CIRCUIT_BYTECODE: *n = BC_N_CONSTRAINTS; return kBytecodeInfo;
    case ZK_CIRCUIT_EVM: *n = EV_N_CONSTRAINTS; return kEvmInfo;
    case ZK_CIRCUIT_COPY: *n = CP_N_CONSTRAINTS; return kCopyInfo;
    case ZK_CIRCUIT_STATE: *n = ST_N_CONSTRAINTS; return kStateInfo;
    case ZK_CIRCUIT_EXP: *n = XP_N_CONSTRAINTS; return kExpInfo;
    case ZK_CIRCUIT_TX: *n = TX_N_CONSTRAINTS; return kTxInfo;
    case ZK_CIRCUIT_SIG: *n = SG_N_CONSTRAINTS; return kSigInfo;
    case ZK_CIRCUIT_PI: *n = PI_N_CONSTRAINTS; return kPiInfo;
    case ZK_CIRCUIT_WITHDRAWAL: *n = WD_N_CONSTRAINTS; return kWdInfo;
    default: *n = 0; return nullptr;
  }
}

// ------------------------------------------------------------------ context
struct Matrix {
  u64* dev = nullptr;
  size_t cap_bytes = 0;
  bool borrowed = false;
  u64 n_rows = 0;
  u32 n_cols = 0;
  unsigned char* flags = nullptr;
  size_t flags_cap = 0;
  u64 flags_rows = 0;
  u64 version = 0;
  const u64* src_offsets = nullptr;   // != nullptr: a bytecode table unrolled by the library from these
  u64 src_contracts = 0;              // (device) contract offsets — regular by construction
  u64 narrow_mask = 0;                // bit c: column c is stored in <= 8 bytes per row, or is a constant below 2^64
  u64 off[ZK_MAX_COLS];               // byte offset of each column inside dev
  unsigned char width[ZK_MAX_COLS];   // bytes per row of each column (fr.cuh:ld_col)
};

struct Index {
  int table_id = -1;
  u32 n_key = 0;
  u32 key_cols[ZK_MAX_KEY];
  u64* slots = nullptr;
  size_t cap = 0;
  u32 pos_kind = ZK_POS_NONE;
  u32* pos_flag = nullptr;  // device flag written by k_pos_verify
  HeadEnt* heads = nullptr;  // ZK_POS_RUNS heads index
  u32* heads_aux = nullptr;  // [ZK_HEADS_CAP] head list, [1] its count, then IndexDev::heads_used: [1] count, [ZK_HEADS_CAP] buckets
  // The hash part (slots) of the index.  Invariant: no kernel probes slots that were not built — a positional table
  // is probed through the slots only when its device flag is 0 (lookup_sync / pos_enabled), and the slots are built
  // whenever that flag is 0.
  enum HashState {
    HASH_BUILT,    // the slots hold the table
    HASH_SKIPPED,  // the flag was read back as 1: not built
    HASH_UNKNOWN,  // the conditional kernels ran (they build iff the device flag is 0)
    HASH_PENDING,  // not built; check_evm reads the flag back and then builds or skips
  } hash = HASH_BUILT;
  u64 built_version = ~0ull;
  u64 built_challenge = ~0ull;
  bool empty_ready = false;  // the slot array is all-empty for an empty table (no per-check memset)
  IndexDev dev;
};

struct ResultBuf {
  u32* first_fail = nullptr;  // device: u32[n] then (8B aligned) u64[n]
  u64* fail_count = nullptr;
  int n = 0;
};

struct zk_ctx {
  int device = 0;
  Matrix circ[ZK_N_CIRCUITS];
  Matrix tab[ZK_N_TABLES];
  Fr chal[ZK_N_CHALLENGES];
  u64 chal_version = 0;
  std::vector<Index*> indexes;
  ResultBuf res[ZK_N_CIRCUITS];
  std::string err;
  u64 launches = 0;
  int sm_count = 148;
  u32* resp_bitmap = nullptr;  // ResponsibleOpcode bitmap of the fixed table (8 KiB)
  u64 resp_bitmap_version = ~0ull;
  unsigned char* stage = nullptr;  // device staging (zk_upload_bytecode_table_from_code)
  size_t stage_cap = 0;
  unsigned char* evm_sort = nullptr;  // EvmSort arrays: bucket[cap] | sorted[cap] | hist, cursor, offs
  size_t evm_sort_cap = 0;
  u32* evm_hist_host = nullptr;  // pinned: histogram read back after k_evm_classify, then the bytecode / rw positional flags
  cudaEvent_t evm_hist_ev = nullptr;
  // the transaction-level group (k_evm_group<TX>: a few thousand threads, each a chain of dependent lookups) runs on its
  // own stream next to the hot kernels; forked after the scatter, joined before the check returns to the caller's stream
  cudaStream_t evm_aux = nullptr;
  cudaEvent_t evm_fork_ev = nullptr, evm_join_ev = nullptr;
  cudaEvent_t evm_index_join_ev = nullptr;  // the rw index's verify on evm_aux is done (check_evm)
  int evm_tx_overlap = -1;  // -1 = not read yet (env ZKCHECK_TX_OVERLAP, default 1)
  int evm_index_overlap = -1;  // -1 = not read yet (env ZKCHECK_INDEX_OVERLAP, default 1): rw verify next to the step sort
  int evm_occ[20] = {0};  // resident blocks per SM of the gate-program kernels (0 = not queried yet)
  std::unordered_map<const void*, int> occ;  // same, row-circuit kernels (keyed by kernel)
  BlockStats* block_stats = nullptr;  // k_evm_block_stats output
  void* state_fold = nullptr;  // k_state_fold output: 64 bytes per resident state row
  size_t state_fold_cap = 0;
  unsigned char* kstage = nullptr;  // zk_keccak256_batch / zk_assign_keccak_table staging
  u32* copy_slow = nullptr;  // copy circuit: [0] = count, [1..] = first rows of the warps deferred to the general kernel
  size_t copy_slow_cap = 0;
  unsigned char* astage = nullptr;  // zk_assign_*: staged inputs + the segmented-scan scratch (chunk values, segment totals)
  size_t astage_cap = 0;
  size_t kstage_cap = 0;
  unsigned char* gather = nullptr;  // zk_allreduce_results: all-gathered result vectors
  size_t gather_cap = 0;
  bool timing = false;
  cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};  // start, after index builds, after check kernel
  cudaStream_t ev_mid_stream = nullptr;
  Fr* wd_rpow = nullptr;  // withdrawal circuit: r^k * 2^64 mod p, k < WD_MAX_RLP, for the challenge in wd_rpow_r
  Fr wd_rpow_r{};
  u64* wd_records = nullptr;  // zk_assign_withdrawal_circuit: staged records
  size_t wd_records_cap = 0;
};
static int mark_indexes_ready(zk_ctx* ctx);

static std::string g_create_err;
static size_t up32(size_t x) { return (x + 31) / 32 * 32; }

#define CK(ctx, call)                                                                  \
  do {                                                                                 \
    cudaError_t e_ = (call);                                                           \
    if (e_ != cudaSuccess) {                                                           \
      (ctx)->err = std::string(#call) + " (api.cu:" + std::to_string(__LINE__) + "): " + cudaGetErrorString(e_); \
      return -2;                                                                       \
    }                                                                                  \
  } while (0)

static int fail_msg(zk_ctx* ctx, const std::string& m) {
  ctx->err = m;
  return -1;
}

extern "C" int zk_ctx_create(int device_ordinal, zk_ctx** out) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    g_create_err = std::string("no CUDA device: ") + cudaGetErrorString(e);
    return -2;
  }
  if (device_ordinal < 0 || device_ordinal >= n) {
    g_create_err = "bad device ordinal";
    return -1;
  }
  e = cudaSetDevice(device_ordinal);
  if (e != cudaSuccess) {
    g_create_err = cudaGetErrorString(e);
    return -2;
  }
  zk_ctx* c = new zk_ctx();
  c->device = device_ordinal;
  cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device_ordinal);
  // defaults: fixed 253-bit constants (callers normally draw their own after fixing the witness)
  c->chal[ZK_CHALLENGE_KECCAK] = Fr{{0x9b97f4a7c15f39ccull, 0x0d6e8feb86659fd9ull, 0x3c2b2ae3d27d4eb4ull, 0x1165667b19e3779full}};
  c->chal[ZK_CHALLENGE_LOOKUP] = Fr{{0x2545f4914f6cdd1dull, 0x5851f42d4c957f2dull, 0x14057b7ef767814full, 0x0fe3a95bd3a1c8e7ull}};
  *out = c;
  return 0;
}

static void free_matrix(Matrix& m) {
  if (m.dev && !m.borrowed) cudaFree(m.dev);
  if (m.flags) cudaFree(m.flags);
  m = Matrix();
}

extern "C" void zk_ctx_destroy(zk_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  for (auto& m : ctx->circ) free_matrix(m);
  for (auto& m : ctx->tab) free_matrix(m);
  for (auto* ix : ctx->indexes) {
    if (ix->slots) cudaFree(ix->slots);
    if (ix->pos_flag) cudaFree(ix->pos_flag);
    if (ix->heads) cudaFree(ix->heads);
    if (ix->heads_aux) cudaFree(ix->heads_aux);
    delete ix;
  }
  if (ctx->stage) cudaFree(ctx->stage);
  for (auto& r : ctx->res)
    if (r.first_fail) cudaFree(r.first_fail);
  for (auto& e : ctx->ev)
    if (e) cudaEventDestroy(e);
  if (ctx->gather) cudaFree(ctx->gather);
  if (ctx->state_fold) cudaFree(ctx->state_fold);
  if (ctx->block_stats) cudaFree(ctx->block_stats);
  if (ctx->evm_sort) cudaFree(ctx->evm_sort);
  if (ctx->kstage) cudaFree(ctx->kstage);
  if (ctx->astage) cudaFree(ctx->astage);
  if (ctx->copy_slow) cudaFree(ctx->copy_slow);
  if (ctx->evm_hist_host) cudaFreeHost(ctx->evm_hist_host);
  if (ctx->evm_hist_ev) cudaEventDestroy(ctx->evm_hist_ev);
  if (ctx->evm_fork_ev) cudaEventDestroy(ctx->evm_fork_ev);
  if (ctx->evm_join_ev) cudaEventDestroy(ctx->evm_join_ev);
  if (ctx->evm_index_join_ev) cudaEventDestroy(ctx->evm_index_join_ev);
  if (ctx->evm_aux) cudaStreamDestroy(ctx->evm_aux);
  if (ctx->resp_bitmap) cudaFree(ctx->resp_bitmap);
  if (ctx->wd_rpow) cudaFree(ctx->wd_rpow);
  if (ctx->wd_records) cudaFree(ctx->wd_records);
  delete ctx;
}

extern "C" const char* zk_last_error(zk_ctx* ctx) {
  return ctx ? ctx->err.c_str() : g_create_err.c_str();
}

static bool fr_is_canonical(const u64 r[4]) {
  Fr a{{r[0], r[1], r[2], r[3]}}, p{{ZK_P0, ZK_P1, ZK_P2, ZK_P3}};
  return fr_lt(a, p);
}

extern "C" int zk_set_challenge(zk_ctx* ctx, int which, const uint64_t r[4]) {
  if (which < 0 || which >= ZK_N_CHALLENGES) return fail_msg(ctx, "bad challenge id");
  if (!fr_is_canonical((const u64*)r)) return fail_msg(ctx, "challenge is not canonical (>= p)");
  ctx->chal[which] = Fr{{r[0], r[1], r[2], r[3]}};
  if (which == ZK_CHALLENGE_LOOKUP) ctx->chal_version++;
  return 0;
}

// `widths` == nullptr: canonical uint64[n_cols][n_rows][4].  Otherwise the packed format of
// include/zkcheck.h: column c holds n_rows integers of widths[c] bytes at byte offset offs[c] of a
// buffer of `total_bytes`; the buffer is copied as it is (one H2D copy) and read in place.
static int store_matrix(zk_ctx* ctx, Matrix& m, u64 n_rows, u32 n_cols, const void* host,
                        const u64* device, cudaStream_t st, const uint8_t* widths = nullptr,
                        const uint64_t* offs = nullptr, size_t total_bytes = 0) {
  CK(ctx, cudaSetDevice(ctx->device));
  if (n_cols > ZK_MAX_COLS) return fail_msg(ctx, "too many columns");
  m.src_offsets = nullptr;
  if (widths) {
    for (u32 c = 0; c < n_cols; c++) {
      const unsigned w = widths[c];
      if (!(w == 0 || w == 1 || w == 2 || w == 4 || w == 8 || w == 16 || w == 32))
        return fail_msg(ctx, "packed column width must be 0, 1, 2, 4, 8, 16 or 32");
      const size_t need = w ? (size_t)w * n_rows : 32;
      if (offs[c] % 32 || offs[c] + need > total_bytes)
        return fail_msg(ctx, "packed column offset misaligned or outside the buffer");
    }
  }
  m.version++;
  if (device) {
    if (m.dev && !m.borrowed) cudaFree(m.dev);
    m.dev = const_cast<u64*>(device);
    m.borrowed = true;
    m.cap_bytes = 0;
  } else {
    size_t bytes = widths ? total_bytes : (size_t)n_rows * n_cols * 32;
    if (m.borrowed) {
      m.dev = nullptr;
      m.borrowed = false;
      m.cap_bytes = 0;
    }
    if (bytes > m.cap_bytes) {
      if (m.dev) cudaFree(m.dev);
      m.dev = nullptr;
      CK(ctx, cudaMalloc(&m.dev, bytes ? bytes : 32));
      m.cap_bytes = bytes;
    }
    if (bytes) CK(ctx, cudaMemcpyAsync(m.dev, host, bytes, cudaMemcpyHostToDevice, st));
  }
  m.n_rows = n_rows;
  m.n_cols = n_cols;
  m.flags_rows = 0;  // flags belong to the previous contents
  m.narrow_mask = 0;
  if (widths) {
    for (u32 c = 0; c < n_cols; c++) {
      m.off[c] = offs[c];
      m.width[c] = widths[c];
      bool narrow = widths[c] >= 1 && widths[c] <= 8;
      if (widths[c] == 0 && host) {  // constant column: narrow iff the one stored cell is below 2^64
        const u64* cell = (const u64*)((const unsigned char*)host + offs[c]);
        narrow = (cell[1] | cell[2] | cell[3]) == 0;
      }
      if (narrow) m.narrow_mask |= 1ull << c;
    }
  } else {
    layout_canonical(m.off, m.width, n_cols, n_rows);
  }
  return 0;
}

static int store_flags(zk_ctx* ctx, Matrix& m, u64 n_rows, const uint8_t* flags, cudaStream_t st) {
  CK(ctx, cudaSetDevice(ctx->device));
  if (n_rows != m.n_rows) return fail_msg(ctx, "flags row count differs from the matrix");
  if (!flags) {
    m.flags_rows = 0;
    return 0;
  }
  if (n_rows > m.flags_cap) {
    if (m.flags) cudaFree(m.flags);
    m.flags = nullptr;
    CK(ctx, cudaMalloc(&m.flags, n_rows ? n_rows : 1));
    m.flags_cap = n_rows;
  }
  CK(ctx, cudaMemcpyAsync(m.flags, flags, n_rows, cudaMemcpyHostToDevice, st));
  m.flags_rows = n_rows;
  return 0;
}

extern "C" int zk_upload_columns(zk_ctx* ctx, int circuit_id, uint64_t n_rows, uint32_t n_cols,
                                 const uint64_t* colmajor, void* stream) {
  if (circuit_id < 0 || circuit_id >= ZK_N_CIRCUITS) return fail_msg(ctx, "bad circuit id");
  if ((int)n_cols != kCircuitCols[circuit_id]) return fail_msg(ctx, "wrong column count for circuit");
  if (n_rows >= 0xFFFFFFFFull) return fail_msg(ctx, "too many rows (row ids are uint32)");
  return store_matrix(ctx, ctx->circ[circuit_id], n_rows, n_cols, (const u64*)colmajor, nullptr,
                      (cudaStream_t)stream);
}
extern "C" int zk_bind_columns_device(zk_ctx* ctx, int circuit_id, uint64_t n_rows, uint32_t n_cols,
                                      const uint64_t* dev) {
  if (circuit_id < 0 || circuit_id >= ZK_N_CIRCUITS) return fail_msg(ctx, "bad circuit id");
  if ((int)n_cols != kCircuitCols[circuit_id]) return fail_msg(ctx, "wrong column count for circuit");
  if (n_rows >= 0xFFFFFFFFull) return fail_msg(ctx, "too many rows (row ids are uint32)");
  return store_matrix(ctx, ctx->circ[circuit_id], n_rows, n_cols, nullptr, (const u64*)dev, 0);
}
extern "C" int zk_upload_row_flags(zk_ctx* ctx, int circuit_id, uint64_t n_rows,
                                   const uint8_t* flags, void* stream) {
  if (circuit_id < 0 || circuit_id >= ZK_N_CIRCUITS) return fail_msg(ctx, "bad circuit id");
  return store_flags(ctx, ctx->circ[circuit_id], n_rows, flags, (cudaStream_t)stream);
}
extern "C" int zk_upload_table(zk_ctx* ctx, int table_id, uint64_t n_rows, uint32_t n_cols,
                               const uint64_t* colmajor, void* stream) {
  if (table_id < 0 || table_id >= ZK_N_TABLES) return fail_msg(ctx, "bad table id");
  if ((int)n_cols != kTableCols[table_id]) return fail_msg(ctx, "wrong column count for table");
  if (n_rows >= 0x7FFFFFFFull) return fail_msg(ctx, "too many table rows");
  return store_matrix(ctx, ctx->tab[table_id], n_rows, n_cols, (const u64*)colmajor, nullptr,
                      (cudaStream_t)stream);
}
extern "C" int zk_bind_table_device(zk_ctx* ctx, int table_id, uint64_t n_rows, uint32_t n_cols,
                                    const uint64_t* dev) {
  if (table_id < 0 || table_id >= ZK_N_TABLES) return fail_msg(ctx, "bad table id");
  if ((int)n_cols != kTableCols[table_id]) return fail_msg(ctx, "wrong column count for table");
  if (n_rows >= 0x7FFFFFFFull) return fail_msg(ctx, "too many table rows");
  return store_matrix(ctx, ctx->tab[table_id], n_rows, n_cols, nullptr, (const u64*)dev, 0);
}
extern "C" int zk_upload_table_flags(zk_ctx* ctx, int table_id, uint64_t n_rows,
                                     const uint8_t* flags, void* stream) {
  if (table_id < 0 || table_id >= ZK_N_TABLES) return fail_msg(ctx, "bad table id");
  return store_flags(ctx, ctx->tab[table_id], n_rows, flags, (cudaStream_t)stream);
}

extern "C" int zk_upload_columns_packed(zk_ctx* ctx, int circuit_id, uint64_t n_rows, uint32_t n_cols,
                                        const void* packed, uint64_t total_bytes, const uint64_t* col_offsets,
                                        const uint8_t* col_widths, void* stream) {
  if (circuit_id < 0 || circuit_id >= ZK_N_CIRCUITS) return fail_msg(ctx, "bad circuit id");
  if ((int)n_cols != kCircuitCols[circuit_id]) return fail_msg(ctx, "wrong column count for circuit");
  if (n_rows >= 0xFFFFFFFFull) return fail_msg(ctx, "too many rows (row ids are uint32)");
  if (!col_offsets || !col_widths) return fail_msg(ctx, "packed upload needs offsets and widths");
  return store_matrix(ctx, ctx->circ[circuit_id], n_rows, n_cols, packed, nullptr, (cudaStream_t)stream, col_widths,
                      col_offsets, (size_t)total_bytes);
}
extern "C" int zk_upload_table_packed(zk_ctx* ctx, int table_id, uint64_t n_rows, uint32_t n_cols,
                                      const void* packed, uint64_t total_bytes, const uint64_t* col_offsets,
                                      const uint8_t* col_widths, void* stream) {
  if (table_id < 0 || table_id >= ZK_N_TABLES) return fail_msg(ctx, "bad table id");
  if ((int)n_cols != kTableCols[table_id]) return fail_msg(ctx, "wrong column count for table");
  if (n_rows >= 0x7FFFFFFFull) return fail_msg(ctx, "too many table rows");
  if (!col_offsets || !col_widths) return fail_msg(ctx, "packed upload needs offsets and widths");
  return store_matrix(ctx, ctx->tab[table_id], n_rows, n_cols, packed, nullptr, (cudaStream_t)stream, col_widths,
                      col_offsets, (size_t)total_bytes);
}

// ------------------------------------------------------------------ bytecode table from code
// Bytecode.table_assignments (typing.py:390-427) on the device: one thread per table row finds its
// contract (binary search over the row starts code_offsets[k] + k) and writes the six cells.
struct BytecodeSrc {
  const unsigned char* code;
  const unsigned char* bits;
  const u64* offsets;  // [n + 1]
  const u64* hashes;   // [n][4]
  u64 n_contracts, n_rows;
};
__global__ void __launch_bounds__(256) k_bytecode_table_expand(BytecodeSrc src, unsigned char* base, const u64 o_hlo,
                                                               const u64 o_hhi, const u64 o_tag, const u64 o_idx,
                                                               const u64 o_isc, const u64 o_val) {
  const u64 stride = (u64)gridDim.x * blockDim.x;
  for (u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x; r < src.n_rows; r += stride) {
    u64 lo = 0, hi = src.n_contracts;  // largest k with offsets[k] + k <= r
    while (hi - lo > 1) {
      const u64 mid = (lo + hi) >> 1;
      if (__ldg(src.offsets + mid) + mid <= r) lo = mid;
      else hi = mid;
    }
    const u64 k = lo, start = __ldg(src.offsets + k), local = r - (start + k);
    ulonglong2 hl, hh;
    hl.x = __ldg(src.hashes + 4 * k);
    hl.y = __ldg(src.hashes + 4 * k + 1);
    hh.x = __ldg(src.hashes + 4 * k + 2);
    hh.y = __ldg(src.hashes + 4 * k + 3);
    ((ulonglong2*)(base + o_hlo))[r] = hl;
    ((ulonglong2*)(base + o_hhi))[r] = hh;
    u32 tag, index, value;
    unsigned char is_code;
    if (local == 0) {  // Header: (hash, Header, 0, 0, len)
      tag = 1;
      index = 0;
      is_code = 0;
      value = (u32)(__ldg(src.offsets + k + 1) - start);
    } else {
      const u64 j = start + local - 1;
      tag = 2;
      index = (u32)(local - 1);
      is_code = (__ldg(src.bits + (j >> 3)) >> (j & 7)) & 1;
      value = __ldg(src.code + j);
    }
    (base + o_tag)[r] = (unsigned char)tag;
    ((u32*)(base + o_idx))[r] = index;
    (base + o_isc)[r] = is_code;
    ((u32*)(base + o_val))[r] = value;
  }
}

extern "C" int zk_upload_bytecode_table_from_code(zk_ctx* ctx, uint64_t n_contracts, const uint8_t* code,
                                                  const uint8_t* is_code_bits, const uint64_t* code_offsets,
                                                  const uint64_t* hashes, void* stream) {
  CK(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  if (n_contracts == 0) return fail_msg(ctx, "no contracts");
  if (code_offsets[0] != 0) return fail_msg(ctx, "code_offsets[0] must be 0");
  for (u64 k = 0; k < n_contracts; k++) {
    if (code_offsets[k + 1] < code_offsets[k]) return fail_msg(ctx, "code_offsets must be non-decreasing");
    if (code_offsets[k + 1] - code_offsets[k] >= 0xFFFFFFFFull) return fail_msg(ctx, "contract too long");
  }
  const u64 total = code_offsets[n_contracts], n_rows = total + n_contracts;
  if (n_rows >= 0x7FFFFFFFull) return fail_msg(ctx, "too many table rows");
  // staging: code | bits | offsets | hashes (each 32-byte aligned)
  const size_t s_code = 0, s_bits = up32(total), s_off = s_bits + up32((total + 7) / 8);
  const size_t s_hash = s_off + up32((n_contracts + 1) * 8), s_total = s_hash + up32(n_contracts * 32);
  if (s_total > ctx->stage_cap) {
    if (ctx->stage) cudaFree(ctx->stage);
    ctx->stage = nullptr;
    CK(ctx, cudaMalloc(&ctx->stage, s_total));
    ctx->stage_cap = s_total;
  }
  unsigned char* sg = ctx->stage;
  if (total) {
    CK(ctx, cudaMemcpyAsync(sg + s_code, code, total, cudaMemcpyHostToDevice, st));
    CK(ctx, cudaMemcpyAsync(sg + s_bits, is_code_bits, (total + 7) / 8, cudaMemcpyHostToDevice, st));
  }
  CK(ctx, cudaMemcpyAsync(sg + s_off, code_offsets, (n_contracts + 1) * 8, cudaMemcpyHostToDevice, st));
  CK(ctx, cudaMemcpyAsync(sg + s_hash, hashes, n_contracts * 32, cudaMemcpyHostToDevice, st));
  // the resident table: packed layout [16, 16, 1, 4, 1, 4]
  static const unsigned char kW[6] = {16, 16, 1, 4, 1, 4};
  Matrix& m = ctx->tab[ZK_TABLE_BYTECODE];
  u64 off[6], bytes = 0;
  for (int c = 0; c < 6; c++) {
    off[c] = bytes;
    bytes += up32((size_t)kW[c] * n_rows);
  }
  if (m.borrowed) {
    m.dev = nullptr;
    m.borrowed = false;
    m.cap_bytes = 0;
  }
  if (bytes > m.cap_bytes) {
    if (m.dev) cudaFree(m.dev);
    m.dev = nullptr;
    CK(ctx, cudaMalloc(&m.dev, bytes));
    m.cap_bytes = bytes;
  }
  m.version++;
  m.n_rows = n_rows;
  m.n_cols = 6;
  m.flags_rows = 0;
  m.src_offsets = (const u64*)(sg + s_off);  // valid until the next call (the staging buffer is reused)
  m.src_contracts = n_contracts;
  for (int c = 0; c < 6; c++) {
    m.off[c] = off[c];
    m.width[c] = kW[c];
  }
  BytecodeSrc src{sg + s_code, sg + s_bits, (const u64*)(sg + s_off), (const u64*)(sg + s_hash), n_contracts, n_rows};
  const unsigned grid = (unsigned)std::min<u64>((n_rows + 255) / 256, (u64)ctx->sm_count * 16);
  k_bytecode_table_expand<<<grid, 256, 0, st>>>(src, (unsigned char*)m.dev, off[0], off[1], off[2], off[3], off[4], off[5]);
  ctx->launches += 1;
  CK(ctx, cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------ Keccak-256 on the device
// The reference hashes on the host through third-party packages (util/hash.py:7-10); witness generators
// call it once per contract / copy event (KeccakCircuit.add, typing.py:854-865; assign_keccak_table,
// bytecode_circuit.py:182-186).  Here one BLOCK takes one message: thread 0 runs the sponge (the
// permutation is sequential), all 128 threads fold the message into its random linear combination
// sum d_i r^(n-1-i) by chunks — Horner inside a chunk, then a shared-memory tree of
// (value, r^length) pairs: value = left * r^len(right) + right.
struct KeccakJob {
  const unsigned char* data;  // all messages concatenated
  const u64* offsets;         // [n + 1]
  u64 n;
};
__global__ void __launch_bounds__(128) k_keccak256(KeccakJob job, u64* digests /* [n][4] lanes */, unsigned char* table, u64 o_tag,
                                                   u64 o_rlc, u64 o_len, u64 o_lo, u64 o_hi, Fr r_mont) {
  __shared__ Fr s_val[128], s_pow[128];
  const u64 m = blockIdx.x;
  if (m >= job.n) return;
  const unsigned char* msg = job.data + job.offsets[m];
  const u64 len = job.offsets[m + 1] - job.offsets[m];
  u64 d[4] = {0, 0, 0, 0};
  if (threadIdx.x == 0) {
    keccak256(msg, len, d);
    if (digests)
      for (int k = 0; k < 4; k++) digests[4 * m + k] = d[k];
  }
  if (!table) return;
  // chunked Horner: thread t owns bytes [t * per, min(len, (t + 1) * per))
  const u64 per = (len + 127) / 128;
  const u64 lo = min(len, threadIdx.x * per), hi = min(len, lo + per);
  rlc_chunk(msg, lo, hi, r_mont, s_val[threadIdx.x], s_pow[threadIdx.x]);
  __syncthreads();
  for (int stride = 1; stride < 128; stride <<= 1) {
    if ((threadIdx.x & (2 * stride - 1)) == 0)
      rlc_combine(s_val[threadIdx.x], s_pow[threadIdx.x], s_val[threadIdx.x + stride], s_pow[threadIdx.x + stride]);
    __syncthreads();
  }
  if (threadIdx.x == 0) {  // the table row (2 = Finalize, input_rlc, input_len, Word(digest as a big-endian integer))
    u64 wlo[2], whi[2];
    keccak_digest_to_word(d, wlo, whi);
    u64* c;
    c = (u64*)(table + o_tag) + 4 * m; c[0] = 2; c[1] = c[2] = c[3] = 0;
    c = (u64*)(table + o_rlc) + 4 * m; for (int k = 0; k < 4; k++) c[k] = s_val[0].l[k];
    c = (u64*)(table + o_len) + 4 * m; c[0] = len; c[1] = c[2] = c[3] = 0;
    c = (u64*)(table + o_lo) + 4 * m; c[0] = wlo[0]; c[1] = wlo[1]; c[2] = c[3] = 0;
    c = (u64*)(table + o_hi) + 4 * m; c[0] = whi[0]; c[1] = whi[1]; c[2] = c[3] = 0;
  }
}
static int keccak_stage(zk_ctx* ctx, uint64_t n, const uint8_t* data, const uint64_t* offsets, cudaStream_t st, KeccakJob* job,
                        u64** dig_dev) {
  if (n == 0) return fail_msg(ctx, "no messages");
  if (offsets[0] != 0) return fail_msg(ctx, "offsets[0] must be 0");
  for (u64 k = 0; k < n; k++)
    if (offsets[k + 1] < offsets[k]) return fail_msg(ctx, "offsets must be non-decreasing");
  const size_t total = offsets[n], s_off = up32(total ? total : 1), s_dig = s_off + up32((n + 1) * 8), s_total = s_dig + n * 32;
  if (s_total > ctx->kstage_cap) {
    if (ctx->kstage) cudaFree(ctx->kstage);
    ctx->kstage = nullptr;
    CK(ctx, cudaMalloc(&ctx->kstage, s_total));
    ctx->kstage_cap = s_total;
  }
  if (total) CK(ctx, cudaMemcpyAsync(ctx->kstage, data, total, cudaMemcpyHostToDevice, st));
  CK(ctx, cudaMemcpyAsync(ctx->kstage + s_off, offsets, (n + 1) * 8, cudaMemcpyHostToDevice, st));
  job->data = ctx->kstage;
  job->offsets = (const u64*)(ctx->kstage + s_off);
  job->n = n;
  *dig_dev = (u64*)(ctx->kstage + s_dig);
  return 0;
}
extern "C" int zk_keccak256_batch(zk_ctx* ctx, uint64_t n, const uint8_t* data, const uint64_t* offsets, uint64_t* digests,
                                  void* stream) {
  CK(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  KeccakJob job;
  u64* dig = nullptr;
  int rc = keccak_stage(ctx, n, data, offsets, st, &job, &dig);
  if (rc) return rc;
  k_keccak256<<<(unsigned)n, 128, 0, st>>>(job, dig, nullptr, 0, 0, 0, 0, 0, Fr{{0, 0, 0, 0}});
  ctx->launches++;
  CK(ctx, cudaGetLastError());
  CK(ctx, cudaMemcpyAsync(digests, dig, n * 32, cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaStreamSynchronize(st));
  return 0;
}
extern "C" int zk_assign_keccak_table(zk_ctx* ctx, uint64_t n, const uint8_t* data, const uint64_t* offsets, void* stream) {
  CK(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  if (n >= 0x7FFFFFFFull) return fail_msg(ctx, "too many table rows");
  KeccakJob job;
  u64* dig = nullptr;
  int rc = keccak_stage(ctx, n, data, offsets, st, &job, &dig);
  if (rc) return rc;
  Matrix& m = ctx->tab[ZK_TABLE_KECCAK];
  const size_t bytes = (size_t)n * 5 * 32;
  if (m.borrowed) {
    m.dev = nullptr;
    m.borrowed = false;
    m.cap_bytes = 0;
  }
  if (bytes > m.cap_bytes) {
    if (m.dev) cudaFree(m.dev);
    m.dev = nullptr;
    CK(ctx, cudaMalloc(&m.dev, bytes));
    m.cap_bytes = bytes;
  }
  m.version++;
  m.n_rows = n;
  m.n_cols = 5;
  m.flags_rows = 0;
  m.src_offsets = nullptr;
  layout_canonical(m.off, m.width, 5, n);
  const Fr r_mont = fr_to_mont(ctx->chal[ZK_CHALLENGE_KECCAK]);
  k_keccak256<<<(unsigned)n, 128, 0, st>>>(job, dig, (unsigned char*)m.dev, m.off[0], m.off[1], m.off[2], m.off[3], m.off[4], r_mont);
  ctx->launches++;
  CK(ctx, cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------ witness assignment on the device (assign.cu)
static int ensure_astage(zk_ctx* ctx, size_t need) {
  if (need > ctx->astage_cap) {
    if (ctx->astage) cudaFree(ctx->astage);
    ctx->astage = nullptr;
    CK(ctx, cudaMalloc(&ctx->astage, need));
    ctx->astage_cap = need;
  }
  return 0;
}
// (re)allocates the resident matrix of a circuit as narrow columns of the given widths
static int alloc_narrow(zk_ctx* ctx, Matrix& m, u64 n_rows, u32 n_cols, const unsigned char* widths, size_t extra_front = 0) {
  size_t bytes = extra_front;
  for (u32 c = 0; c < n_cols; c++) {
    m.off[c] = bytes;
    m.width[c] = widths[c];
    bytes += up32((size_t)widths[c] * n_rows);
  }
  if (m.borrowed) {
    m.dev = nullptr;
    m.borrowed = false;
    m.cap_bytes = 0;
  }
  if (bytes > m.cap_bytes) {
    if (m.dev) cudaFree(m.dev);
    m.dev = nullptr;
    CK(ctx, cudaMalloc(&m.dev, bytes ? bytes : 32));
    m.cap_bytes = bytes;
  }
  m.version++;
  m.n_rows = n_rows;
  m.n_cols = n_cols;
  m.flags_rows = 0;
  m.src_offsets = nullptr;
  m.narrow_mask = 0;
  return 0;
}
// chunk table of a segmented Horner scan: ceil(len / 32) chunks per segment
static std::vector<u64> chunk_offsets(const u64* seg_off, u64 n_seg) {
  std::vector<u64> c(n_seg + 1, 0);
  for (u64 k = 0; k < n_seg; k++) c[k + 1] = c[k] + (seg_off[k + 1] - seg_off[k] + ZK_SEG_CHUNK - 1) / ZK_SEG_CHUNK;
  return c;
}
static int run_seg_scan(zk_ctx* ctx, const SegHorner& s, Fr* chunk_val, Fr* seg_total, cudaStream_t st) {
  if (s.n_chunks == 0) return 0;
  k_seg_local<<<(unsigned)((s.n_chunks + 255) / 256), 256, 0, st>>>(s, chunk_val);
  k_seg_carry<<<(unsigned)((s.n_seg + 127) / 128), 128, 0, st>>>(s, chunk_val, seg_total);
  ctx->launches += 2;
  CK(ctx, cudaGetLastError());
  return 0;
}

extern "C" int zk_assign_bytecode_circuit(zk_ctx* ctx, uint32_t k, uint64_t n_contracts, const uint8_t* code,
                                          const uint8_t* is_code_bits, const uint64_t* code_offsets, const uint64_t* hashes,
                                          void* stream) {
  CK(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  if (k > 31) return fail_msg(ctx, "2^k rows: k must be <= 31 (row ids are uint32)");
  if (n_contracts == 0) return fail_msg(ctx, "no contracts");
  if (code_offsets[0] != 0) return fail_msg(ctx, "code_offsets[0] must be 0");
  for (u64 c = 0; c < n_contracts; c++) {
    if (code_offsets[c + 1] < code_offsets[c]) return fail_msg(ctx, "code_offsets must be non-decreasing");
    if (code_offsets[c + 1] - code_offsets[c] >= 0xFFFFFFFFull) return fail_msg(ctx, "contract too long");
  }
  const u64 total = code_offsets[n_contracts], n_rows = 1ull << k;
  const std::vector<u64> chunks = chunk_offsets((const u64*)code_offsets, n_contracts);
  const u64 n_chunks = chunks[n_contracts];
  const size_t s_code = 0, s_bits = up32(total), s_off = s_bits + up32((total + 7) / 8), s_chk = s_off + up32((n_contracts + 1) * 8);
  const size_t s_hash = s_chk + up32((n_contracts + 1) * 8), s_val = s_hash + up32(n_contracts * 32), s_total = s_val + (n_chunks + 1) * 32;
  int rc;
  if ((rc = ensure_astage(ctx, s_total))) return rc;
  unsigned char* sg = ctx->astage;
  if (total) {
    CK(ctx, cudaMemcpyAsync(sg + s_code, code, total, cudaMemcpyHostToDevice, st));
    CK(ctx, cudaMemcpyAsync(sg + s_bits, is_code_bits, (total + 7) / 8, cudaMemcpyHostToDevice, st));
  }
  CK(ctx, cudaMemcpyAsync(sg + s_off, code_offsets, (n_contracts + 1) * 8, cudaMemcpyHostToDevice, st));
  CK(ctx, cudaMemcpyAsync(sg + s_chk, chunks.data(), (n_contracts + 1) * 8, cudaMemcpyHostToDevice, st));
  CK(ctx, cudaMemcpyAsync(sg + s_hash, hashes, n_contracts * 32, cudaMemcpyHostToDevice, st));
  Matrix& m = ctx->circ[ZK_CIRCUIT_BYTECODE];
  if ((rc = alloc_narrow(ctx, m, n_rows, 12, kBytecodeAssignWidths))) return rc;
  BytecodeAssign a;
  a.s = SegHorner{sg + s_code, (const u64*)(sg + s_off), (const u64*)(sg + s_chk), n_contracts, n_chunks,
                  fr_to_mont(ctx->chal[ZK_CHALLENGE_KECCAK])};
  a.bits = sg + s_bits;
  a.hashes = (const u64*)(sg + s_hash);
  a.n_rows = n_rows;
  a.n_table_rows = total + n_contracts;
  a.base = (unsigned char*)m.dev;
  for (int c = 0; c < 12; c++) a.off[c] = m.off[c];
  Fr* chunk_val = (Fr*)(sg + s_val);
  if ((rc = run_seg_scan(ctx, a.s, chunk_val, nullptr, st))) return rc;
  k_assign_bytecode_rows<<<(unsigned)std::min<u64>((n_rows + 255) / 256, (u64)ctx->sm_count * 16), 256, 0, st>>>(a);
  if (n_chunks) k_assign_bytecode_rlc<<<(unsigned)((n_chunks + 255) / 256), 256, 0, st>>>(a, chunk_val);
  ctx->launches += n_chunks ? 2 : 1;
  CK(ctx, cudaGetLastError());
  return 0;
}

extern "C" int zk_assign_state_circuit(zk_ctx* ctx, uint64_t n_rows, const void* packed_ops, uint64_t total_bytes,
                                       const uint64_t* col_offsets, const uint8_t* col_widths, const uint8_t* row_flags,
                                       void* stream) {
  CK(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  if (n_rows >= 0xFFFFFFFFull) return fail_msg(ctx, "too many rows (row ids are uint32)");
  if (!col_offsets || !col_widths) return fail_msg(ctx, "zk_assign_state_circuit needs offsets and widths of the 15 operation columns");
  for (int c = 0; c < 15; c++) {
    const unsigned w = col_widths[c];
    if (!(w == 0 || w == 1 || w == 2 || w == 4 || w == 8 || w == 16 || w == 32)) return fail_msg(ctx, "packed column width must be 0, 1, 2, 4, 8, 16 or 32");
    if (col_offsets[c] % 32 || col_offsets[c] + (w ? (size_t)w * n_rows : 32) > total_bytes)
      return fail_msg(ctx, "packed column offset misaligned or outside the buffer");
  }
  if (col_widths[4] == 32) {  // op.address.to_bytes(20, "little") raises OverflowError beyond 160 bits (state_circuit.py:832)
    const u64* a = (const u64*)((const unsigned char*)packed_ops + col_offsets[4]);
    for (u64 r = 0; r < n_rows; r++)
      if ((a[4 * r + 2] >> 32) || a[4 * r + 3]) return fail_msg(ctx, "operation address does not fit 20 bytes (op2row raises OverflowError)");
  }
  // resident buffer: [uploaded operation columns | 10 limb columns (u16) | 32 key-byte columns (u8)]
  Matrix& m = ctx->circ[ZK_CIRCUIT_STATE];
  const size_t front = up32(total_bytes), limb_stride = up32(2 * n_rows), byte_stride = up32(n_rows);
  const size_t bytes = front + 10 * limb_stride + 32 * byte_stride;
  if (m.borrowed) {
    m.dev = nullptr;
    m.borrowed = false;
    m.cap_bytes = 0;
  }
  if (bytes > m.cap_bytes) {
    if (m.dev) cudaFree(m.dev);
    m.dev = nullptr;
    CK(ctx, cudaMalloc(&m.dev, bytes ? bytes : 32));
    m.cap_bytes = bytes;
  }
  if (total_bytes) CK(ctx, cudaMemcpyAsync(m.dev, packed_ops, total_bytes, cudaMemcpyHostToDevice, st));
  m.version++;
  m.n_rows = n_rows;
  m.n_cols = 57;
  m.src_offsets = nullptr;
  for (int c = 0; c < 8; c++) m.off[c] = col_offsets[c], m.width[c] = col_widths[c];
  for (int q = 0; q < 10; q++) m.off[8 + q] = front + q * limb_stride, m.width[8 + q] = 2;
  for (int q = 0; q < 32; q++) m.off[18 + q] = front + 10 * limb_stride + q * byte_stride, m.width[18 + q] = 1;
  for (int c = 8; c < 15; c++) m.off[42 + c] = col_offsets[c], m.width[42 + c] = col_widths[c];
  int rc;
  if ((rc = store_flags(ctx, m, n_rows, row_flags, st))) return rc;
  if (n_rows == 0) return 0;
  StateAssign a;
  a.base = (const unsigned char*)m.dev;
  a.off_addr = col_offsets[4], a.off_klo = col_offsets[6], a.off_khi = col_offsets[7];
  a.w_addr = col_widths[4], a.w_klo = col_widths[6], a.w_khi = col_widths[7];
  a.limbs = (unsigned char*)m.dev + front;
  a.kbytes = (unsigned char*)m.dev + front + 10 * limb_stride;
  a.n_rows = n_rows, a.limb_stride = limb_stride, a.byte_stride = byte_stride;
  k_assign_state_derive<<<(unsigned)std::min<u64>((n_rows + 255) / 256, (u64)ctx->sm_count * 16), 256, 0, st>>>(a);
  ctx->launches++;
  CK(ctx, cudaGetLastError());
  return 0;
}

extern "C" int zk_assign_copy_circuit(zk_ctx* ctx, uint64_t n_events, const uint64_t* events, const uint8_t* data,
                                      const uint8_t* is_code_bits, void* stream) {
  CK(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  static_assert(sizeof(CopyEvent) == 16 * sizeof(u64), "CopyEvent is 16 u64");
  std::vector<u64> seg(n_events + 1, 0);
  for (u64 e = 0; e < n_events; e++) seg[e + 1] = seg[e] + events[16 * e + 5];
  const u64 total = seg[n_events], n_rows = 2 * total;
  if (n_rows >= 0xFFFFFFFFull) return fail_msg(ctx, "too many rows (row ids are uint32)");
  const std::vector<u64> chunks = chunk_offsets(seg.data(), n_events);
  const u64 n_chunks = chunks[n_events];
  const size_t s_data = 0, s_bits = up32(total), s_off = s_bits + up32((total + 7) / 8), s_chk = s_off + up32((n_events + 1) * 8);
  const size_t s_ev = s_chk + up32((n_events + 1) * 8), s_val = s_ev + up32(n_events * sizeof(CopyEvent));
  const size_t s_tot = s_val + (n_chunks + 1) * 32, s_total = s_tot + (n_events + 1) * 32;
  int rc;
  if ((rc = ensure_astage(ctx, s_total))) return rc;
  unsigned char* sg = ctx->astage;
  if (total) {
    CK(ctx, cudaMemcpyAsync(sg + s_data, data, total, cudaMemcpyHostToDevice, st));
    if (is_code_bits) CK(ctx, cudaMemcpyAsync(sg + s_bits, is_code_bits, (total + 7) / 8, cudaMemcpyHostToDevice, st));
  }
  CK(ctx, cudaMemcpyAsync(sg + s_off, seg.data(), (n_events + 1) * 8, cudaMemcpyHostToDevice, st));
  CK(ctx, cudaMemcpyAsync(sg + s_chk, chunks.data(), (n_events + 1) * 8, cudaMemcpyHostToDevice, st));
  if (n_events) CK(ctx, cudaMemcpyAsync(sg + s_ev, events, n_events * sizeof(CopyEvent), cudaMemcpyHostToDevice, st));
  Matrix& m = ctx->circ[ZK_CIRCUIT_COPY];
  if ((rc = alloc_narrow(ctx, m, n_rows, 20, kCopyAssignWidths))) return rc;
  if (n_rows > m.flags_cap) {
    if (m.flags) cudaFree(m.flags);
    m.flags = nullptr;
    CK(ctx, cudaMalloc(&m.flags, n_rows));
    m.flags_cap = n_rows;
  }
  m.flags_rows = n_rows;
  if (n_chunks == 0) return 0;
  CopyAssign a;
  a.s = SegHorner{sg + s_data, (const u64*)(sg + s_off), (const u64*)(sg + s_chk), n_events, n_chunks,
                  fr_to_mont(ctx->chal[ZK_CHALLENGE_KECCAK])};
  a.ev = (const CopyEvent*)(sg + s_ev);
  a.bits = is_code_bits ? sg + s_bits : nullptr;
  a.base = (unsigned char*)m.dev;
  a.flags = m.flags;
  for (int c = 0; c < 20; c++) a.off[c] = m.off[c];
  a.n_rows = n_rows;
  Fr* chunk_val = (Fr*)(sg + s_val);
  Fr* seg_total = (Fr*)(sg + s_tot);
  if ((rc = run_seg_scan(ctx, a.s, chunk_val, seg_total, st))) return rc;
  k_assign_copy_rows<<<(unsigned)((n_chunks + 255) / 256), 256, 0, st>>>(a, chunk_val, seg_total);
  ctx->launches++;
  CK(ctx, cudaGetLastError());
  return 0;
}

extern "C" int64_t zk_resident_rows(zk_ctx* ctx, int circuit_id) {
  if (circuit_id < 0 || circuit_id >= ZK_N_CIRCUITS) return -1;
  return (int64_t)ctx->circ[circuit_id].n_rows;
}

// the resident matrix of a circuit widened back to canonical cells on the host (inspection / tests)
extern "C" int zk_download_columns(zk_ctx* ctx, int circuit_id, uint64_t* colmajor_out, uint8_t* flags_out, void* stream) {
  if (circuit_id < 0 || circuit_id >= ZK_N_CIRCUITS) return fail_msg(ctx, "bad circuit id");
  CK(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  const Matrix& m = ctx->circ[circuit_id];
  CK(ctx, cudaStreamSynchronize(st));
  std::vector<unsigned char> tmp;
  for (u32 c = 0; c < m.n_cols; c++) {
    const unsigned w = m.width[c];
    const size_t nb = w ? (size_t)w * m.n_rows : 32;
    tmp.resize(nb);
    if (m.n_rows) CK(ctx, cudaMemcpy(tmp.data(), (const unsigned char*)m.dev + m.off[c], nb, cudaMemcpyDeviceToHost));
    u64* out = (u64*)colmajor_out + (size_t)c * m.n_rows * 4;
    for (u64 r = 0; r < m.n_rows; r++) {
      u64 v[4] = {0, 0, 0, 0};
      memcpy(v, tmp.data() + (w ? (size_t)w * r : 0), w ? w : 32);
      memcpy(out + 4 * r, v, 32);
    }
  }
  if (flags_out) {
    if (m.flags_rows == m.n_rows && m.n_rows) CK(ctx, cudaMemcpy(flags_out, m.flags, m.n_rows, cudaMemcpyDeviceToHost));
    else memset(flags_out, 0, m.n_rows);
  }
  return 0;
}

// ------------------------------------------------------------------ lookup index cache
static TableDev table_dev(const zk_ctx* ctx, int table_id) {
  const Matrix& m = ctx->tab[table_id];
  TableDev t;
  t.base = (const unsigned char*)m.dev;
  t.n_rows = m.dev ? m.n_rows : 0;
  t.n_cols = m.n_cols ? m.n_cols : kTableCols[table_id];
  for (u32 c = 0; c < ZK_MAX_TABLE_COLS; c++) {
    t.off[c] = c < t.n_cols && m.dev ? m.off[c] : 0;
    t.width[c] = c < t.n_cols && m.dev ? m.width[c] : 32;
  }
  t.flags = (m.flags_rows == m.n_rows && m.n_rows) ? m.flags : nullptr;
  return t;
}


// persistent grid: no more blocks than the device keeps resident (occupancy x SMs); threads walk the
// rows with a grid stride
template <class K>
static unsigned grid_persistent(zk_ctx* ctx, K kernel, int threads, u64 n_items) {
  const void* key = (const void*)kernel;
  auto it = ctx->occ.find(key);
  if (it == ctx->occ.end()) {
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, threads, 0) != cudaSuccess || occ < 1) occ = 1;
    it = ctx->occ.emplace(key, occ).first;
  }
  const u64 want = (n_items + threads - 1) / threads;
  return (unsigned)std::max<u64>(1, std::min<u64>(want, (u64)it->second * ctx->sm_count));
}
#define ZK_HEADS_CAP (1u << 16)
// The index of `table_id` on `key_cols` (created on first use; a ZK_POS_RUNS index starts with an all-free heads index)
static int find_index(zk_ctx* ctx, int table_id, const u32* key_cols, u32 n_key, u32 pos_kind, cudaStream_t st, Index** out) {
  if (n_key == 0 || n_key > ZK_MAX_KEY) return fail_msg(ctx, "bad key width");
  Index* ix = nullptr;
  for (auto* c : ctx->indexes)
    if (c->table_id == table_id && c->n_key == n_key && !memcmp(c->key_cols, key_cols, 4 * n_key)) ix = c;
  if (!ix) {
    ix = new Index();
    ix->table_id = table_id;
    ix->n_key = n_key;
    memcpy(ix->key_cols, key_cols, 4 * n_key);
    ix->pos_kind = pos_kind;
    ctx->indexes.push_back(ix);
    if (pos_kind != ZK_POS_NONE) {
      CK(ctx, cudaMalloc(&ix->pos_flag, 2 * sizeof(u32)));
      if (pos_kind == ZK_POS_RUNS) {
        CK(ctx, cudaMalloc(&ix->heads, ZK_HEADS_CAP * sizeof(HeadEnt)));
        CK(ctx, cudaMalloc(&ix->heads_aux, (2 * ZK_HEADS_CAP + 2) * sizeof(u32)));
        CK(ctx, cudaMemsetAsync(ix->heads, 0xFF, ZK_HEADS_CAP * sizeof(HeadEnt), st));
        CK(ctx, cudaMemsetAsync(ix->heads_aux, 0, (2 * ZK_HEADS_CAP + 2) * sizeof(u32), st));
      }
    }
  }
  *out = ix;
  return 0;
}
static bool index_current(const zk_ctx* ctx, const Index* ix) {
  return ix->built_version == ctx->tab[ix->table_id].version && ix->built_challenge == ctx->chal_version;
}
// Fill ix->dev for the resident table and lookup challenge (host only; grows the slot array if needed)
static int describe_index(zk_ctx* ctx, Index* ix) {
  const int table_id = ix->table_id;
  const u32 n_key = ix->n_key;
  const u32* key_cols = ix->key_cols;
  TableDev t = table_dev(ctx, table_id);
  size_t cap = 64;
  while (cap < 2 * t.n_rows) cap <<= 1;
  if (cap > ix->cap) {
    if (ix->slots) cudaFree(ix->slots);
    ix->slots = nullptr;
    CK(ctx, cudaMalloc(&ix->slots, cap * sizeof(u64)));
    ix->cap = cap;
    ix->empty_ready = false;
  }
  IndexDev& d = ix->dev;
  d.tab = t;
  d.slots = ix->slots;
  d.mask = (u32)(ix->cap - 1);
  d.n_key = n_key;
  // hash keys: a splitmix64 stream seeded by the lookup challenge
  {
    const Fr& c = ctx->chal[ZK_CHALLENGE_LOOKUP];
    u64 x = c.l[0] ^ (c.l[1] * 0x9E3779B97F4A7C15ull) ^ (c.l[2] * 0xC2B2AE3D27D4EB4Full) ^ (c.l[3] * 0x165667B19E3779F9ull);
    auto next = [&x]() {
      x += 0x9E3779B97F4A7C15ull;
      u64 z = x;
      z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
      z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
      return z ^ (z >> 31);
    };
    for (int k = 0; k < 4; k++) d.hk[k] = next() | 1ull;
    for (u32 j = 0; j < ZK_MAX_KEY; j++) {
      d.key_cols[j] = j < n_key ? key_cols[j] : 0;
      d.hm[j] = next() | 1ull;
    }
  }
  d.pos_kind = ix->pos_kind;
  // lookups go positional only if the table is not empty (an empty table's flag is never initialised)
  d.pos_ok = (t.n_rows && ix->pos_kind != ZK_POS_NONE) ? ix->pos_flag : nullptr;
  // the rw table may end in a run of `Start` padding rows (tag column 2 == Target.Start == 1)
  d.tail_key = -1;
  d.tail_col = d.tail_val = 0;
  if (table_id == ZK_TABLE_RW && ix->pos_kind == ZK_POS_DENSE) {
    d.tail_col = 2;
    d.tail_val = 1;
    for (u32 j = 0; j < n_key; j++)
      if (key_cols[j] == 2) d.tail_key = (int)j;
  }
  d.heads = ix->heads;
  d.heads_mask = ZK_HEADS_CAP - 1;
  d.heads_list = ix->heads_aux;
  d.heads_count = ix->heads_aux ? ix->heads_aux + ZK_HEADS_CAP : nullptr;
  d.heads_used = ix->heads_aux ? ix->heads_aux + ZK_HEADS_CAP + 1 : nullptr;
  return 0;
}
// one k_pos_prep launch for the positional indexes about to be verified (non-empty tables)
static int launch_pos_prep(zk_ctx* ctx, Index* const* ixs, u32 n, cudaStream_t st) {
  if (n == 0) return 0;
  if (n > ZK_POS_PREP_MAX) return fail_msg(ctx, "k_pos_prep: too many indexes");
  PosPrep p{};
  p.n = n;
  p.heads_cap = ZK_HEADS_CAP;
  for (u32 e = 0; e < n; e++) {
    const IndexDev& d = ixs[e]->dev;
    p.flag[e] = ixs[e]->pos_flag;
    p.n_rows[e] = (u32)d.tab.n_rows;
    p.heads[e] = d.heads;
    p.heads_count[e] = d.heads_count;
    p.heads_used[e] = d.heads_used;
  }
  k_pos_prep<<<1, 1024, 0, st>>>(p);
  ctx->launches++;
  CK(ctx, cudaGetLastError());
  return 0;
}
// the structure verify of a positional index over a non-empty table (after its k_pos_prep); the flag stays 1 iff it holds
static int launch_pos_verify(zk_ctx* ctx, Index* ix, cudaStream_t st) {
  const IndexDev& d = ix->dev;
  const Matrix& m = ctx->tab[ix->table_id];
  const u64 n = d.tab.n_rows;
  if (ix->pos_kind == ZK_POS_RUNS && m.src_offsets) {
    // unrolled by the library: regular by construction, heads + lengths straight from the offsets
    k_heads_from_offsets<<<(unsigned)std::min<u64>((m.src_contracts + 255) / 256, 64), 256, 0, st>>>(
        d, ix->pos_flag, m.src_offsets, m.src_contracts);
    ctx->launches++;
  } else if (ix->pos_kind == ZK_POS_DENSE) {
    // the typed strip form for a narrow counter (4 / 8 bytes) and a narrow tail column (1 byte or a constant cell)
    const u32 kc = d.key_cols[0], tc = d.tail_col;
    const unsigned char* pc = d.tab.base + d.tab.off[kc];
    const unsigned char* pt = d.tab.base + d.tab.off[tc];
    const int wc = d.tab.width[kc], wt = d.tail_key >= 0 ? d.tab.width[tc] : 0;
    const bool typed = ((m.narrow_mask >> kc) & 1) && (wc == 4 || wc == 8) && ((uintptr_t)pc & 15) == 0 &&
                       (d.tail_key < 0 || (((m.narrow_mask >> tc) & 1) && (wt == 0 || (wt == 1 && ((uintptr_t)pt & 7) == 0))));
    if (typed) {
      const u64 strips = (n + ZK_DENSE_STRIP - 1) / ZK_DENSE_STRIP;
      const unsigned g = (unsigned)std::min<u64>((strips + 255) / 256, (u64)ctx->sm_count * 16);
      if (wc == 4 && wt == 0) k_pos_verify_dense_typed<4, 0><<<g, 256, 0, st>>>(d, ix->pos_flag);
      else if (wc == 4) k_pos_verify_dense_typed<4, 1><<<g, 256, 0, st>>>(d, ix->pos_flag);
      else if (wt == 0) k_pos_verify_dense_typed<8, 0><<<g, 256, 0, st>>>(d, ix->pos_flag);
      else k_pos_verify_dense_typed<8, 1><<<g, 256, 0, st>>>(d, ix->pos_flag);
    } else {
      k_pos_verify<<<(unsigned)std::min<u64>((n + 255) / 256, (u64)ctx->sm_count * 32), 256, 0, st>>>(d, ix->pos_flag);
    }
    ctx->launches++;
  } else {
    k_pos_verify<<<(unsigned)std::min<u64>((n + 255) / 256, (u64)ctx->sm_count * 32), 256, 0, st>>>(d, ix->pos_flag);
    k_pos_runlen<<<16, 256, 0, st>>>(d);  // run lengths from the listed heads (a few thousand threads at most)
    ctx->launches += 2;
  }
  CK(ctx, cudaGetLastError());
  return 0;
}
// the generic hash index over a non-empty table; `conditional`: both kernels return at once when the positional flag is
// set (the flag is not known on the host)
static int launch_hash_build(zk_ctx* ctx, Index* ix, cudaStream_t st, bool conditional) {
  const IndexDev& d = ix->dev;
  k_slots_clear<<<grid_persistent(ctx, k_slots_clear, 256, ix->cap), 256, 0, st>>>(ix->slots, ix->cap, conditional ? d.pos_ok : nullptr);
  k_index_build<<<grid_persistent(ctx, k_index_build, 256, d.tab.n_rows), 256, 0, st>>>(d);
  ctx->launches += 2;
  CK(ctx, cudaGetLastError());
  ix->hash = !conditional || !d.pos_ok ? Index::HASH_BUILT : Index::HASH_UNKNOWN;
  return 0;
}
// After the positional part (if any) is enqueued: the hash part, or (`defer_hash`, positional tables) nothing yet —
// the caller reads the flag back and calls resolve_hash.
static int finish_index(zk_ctx* ctx, Index* ix, cudaStream_t st, bool defer_hash) {
  const IndexDev& d = ix->dev;
  int rc;
  if (d.tab.n_rows) {
    if (d.pos_ok && defer_hash) ix->hash = Index::HASH_PENDING;
    else if ((rc = launch_hash_build(ctx, ix, st, d.pos_ok != nullptr))) return rc;
  } else {
    if (!ix->empty_ready) CK(ctx, cudaMemsetAsync(ix->slots, 0xFF, ix->cap * sizeof(u64), st));  // once per slot array
    ix->hash = Index::HASH_BUILT;
  }
  ix->empty_ready = d.tab.n_rows == 0;
  ix->built_version = ctx->tab[ix->table_id].version;
  ix->built_challenge = ctx->chal_version;
  return 0;
}
// a pending hash part once the host knows the flag: built iff the table is not positional
static int resolve_hash(zk_ctx* ctx, Index* ix, bool positional, cudaStream_t st) {
  if (ix->hash != Index::HASH_PENDING) return 0;
  if (positional) {
    ix->hash = Index::HASH_SKIPPED;
    return 0;
  }
  return launch_hash_build(ctx, ix, st, false);
}

// Returns the device descriptor of the index of `table_id` on `key_cols`, building it on
// `st` if the table or the lookup challenge changed since the last build.
static int ensure_index(zk_ctx* ctx, int table_id, const u32* key_cols, u32 n_key, cudaStream_t st,
                        IndexDev* out, u32 pos_kind = ZK_POS_NONE) {
  Index* ix = nullptr;
  int rc;
  if ((rc = find_index(ctx, table_id, key_cols, n_key, pos_kind, st, &ix))) return rc;
  if (index_current(ctx, ix)) {
    ix->dev.tab = table_dev(ctx, table_id);  // flags may have been (re)uploaded
    // left pending by an EVM check that did not get to read its flag back
    if (ix->hash == Index::HASH_PENDING && (rc = launch_hash_build(ctx, ix, st, true))) return rc;
    *out = ix->dev;
    return 0;
  }
  if ((rc = describe_index(ctx, ix))) return rc;
  if (ix->dev.pos_ok) {
    if ((rc = launch_pos_prep(ctx, &ix, 1, st))) return rc;
    if ((rc = launch_pos_verify(ctx, ix, st))) return rc;
  }
  if ((rc = finish_index(ctx, ix, st, false))) return rc;
  *out = ix->dev;
  return 0;
}

extern "C" int zk_invalidate_indexes(zk_ctx* ctx) {
  // the fixed table is a circuit constant (uploaded once): its index, like its ResponsibleOpcode
  // bitmap, lives until the table is uploaded again
  for (auto* ix : ctx->indexes)
    if (ix->table_id != ZK_TABLE_FIXED) ix->built_version = ~0ull;
  return 0;
}

// ------------------------------------------------------------------ results
static int ensure_result(zk_ctx* ctx, int circuit, ResultDev* out, cudaStream_t st) {
  int n = 0;
  circuit_info(circuit, &n);
  if (n == 0) return fail_msg(ctx, "circuit has no gate program in this build");
  ResultBuf& r = ctx->res[circuit];
  if (!r.first_fail) {
    size_t off = ((size_t)n * 4 + 7) & ~(size_t)7;
    void* p = nullptr;
    CK(ctx, cudaMalloc(&p, off + (size_t)n * 8));
    r.first_fail = (u32*)p;
    r.fail_count = (u64*)((char*)p + off);
    r.n = n;
  }
  CK(ctx, cudaMemsetAsync(r.first_fail, 0xFF, (size_t)n * 4, st));
  CK(ctx, cudaMemsetAsync(r.fail_count, 0, (size_t)n * 8, st));
  out->first_fail = r.first_fail;
  out->fail_count = r.fail_count;
  return 0;
}

static WitnessDev witness_dev(const Matrix& m) {
  WitnessDev w;
  w.base = (const unsigned char*)m.dev;
  w.n_rows = m.n_rows;
  for (u32 c = 0; c < ZK_MAX_COLS; c++) {
    w.off[c] = c < m.n_cols ? m.off[c] : 0;
    w.width[c] = c < m.n_cols ? m.width[c] : 32;
  }
  w.flags = (m.flags_rows == m.n_rows && m.n_rows) ? m.flags : nullptr;
  return w;
}

// ------------------------------------------------------------------ dispatch
static bool is_canonical(const Matrix& m) {
  for (u32 c = 0; c < m.n_cols; c++)
    if (m.width[c] != 32) return false;
  return true;
}
static int check_bytecode(zk_ctx* ctx, const CheckRange& rg, ResultDev res, cudaStream_t st) {
  const u32 pk[2] = {0, 1}, kk[5] = {0, 1, 2, 3, 4};
  IndexDev push_ix, kec_ix;
  int rc;
  if ((rc = ensure_index(ctx, ZK_TABLE_PUSH, pk, 2, st, &push_ix, ZK_POS_DENSE))) return rc;
  if ((rc = ensure_index(ctx, ZK_TABLE_KECCAK, kk, 5, st, &kec_ix))) return rc;
  if ((rc = mark_indexes_ready(ctx))) return rc;
  const u64 n = rg.row_end - rg.row_begin;
  const Fr r_mont = fr_to_mont(ctx->chal[ZK_CHALLENGE_KECCAK]);
  const Matrix& m = ctx->circ[ZK_CIRCUIT_BYTECODE];
  if (is_canonical(m))
    k_check_bytecode<L_CANON><<<grid_persistent(ctx, k_check_bytecode<L_CANON>, 256, n), 256, 0, st>>>(witness_dev(m), rg, push_ix, kec_ix, r_mont, res);
  else
    k_check_bytecode<L_ANY><<<grid_persistent(ctx, k_check_bytecode<L_ANY>, 256, n), 256, 0, st>>>(witness_dev(m), rg, push_ix, kec_ix, r_mont, res);
  ctx->launches++;
  CK(ctx, cudaGetLastError());
  return 0;
}

static int check_tx(zk_ctx* ctx, const CheckRange& rg, ResultDev res, cudaStream_t st, bool sig = false) {
  const u32 kk[5] = {0, 1, 2, 3, 4};
  IndexDev kec_ix;
  int rc;
  if ((rc = ensure_index(ctx, ZK_TABLE_KECCAK, kk, 5, st, &kec_ix))) return rc;
  if ((rc = mark_indexes_ready(ctx))) return rc;
  const u64 n = rg.row_end - rg.row_begin;
  const unsigned grid = (unsigned)std::min<u64>((n + 127) / 128, (u64)ctx->sm_count * 16);
  const Fr r_mont = fr_to_mont(ctx->chal[ZK_CHALLENGE_KECCAK]);
  if (sig) k_check_sig<<<grid, 128, 0, st>>>(witness_dev(ctx->circ[ZK_CIRCUIT_SIG]), rg, kec_ix, r_mont, res);
  else k_check_tx<<<grid, 128, 0, st>>>(witness_dev(ctx->circ[ZK_CIRCUIT_TX]), rg, kec_ix, r_mont, res);
  ctx->launches++;
  CK(ctx, cudaGetLastError());
  return 0;
}

static int check_exp(zk_ctx* ctx, const CheckRange& rg, ResultDev res, cudaStream_t st) {
  const Matrix& m = ctx->circ[ZK_CIRCUIT_EXP];
  if (!(rg.flags & ZK_FLAG_WRAP) && rg.row_end + 1 > m.n_rows)
    return fail_msg(ctx, "exp rows [b,e) need row e resident (rotation +1) unless ZK_FLAG_WRAP");
  int rc;
  if ((rc = mark_indexes_ready(ctx))) return rc;
  const u64 n = rg.row_end - rg.row_begin;
  if (is_canonical(m)) k_check_exp<L_CANON><<<grid_persistent(ctx, k_check_exp<L_CANON>, 128, n), 128, 0, st>>>(witness_dev(m), rg, res);
  else k_check_exp<L_ANY><<<grid_persistent(ctx, k_check_exp<L_ANY>, 128, n), 128, 0, st>>>(witness_dev(m), rg, res);
  ctx->launches++;
  CK(ctx, cudaGetLastError());
  return 0;
}

static int check_pi(zk_ctx* ctx, const CheckRange& rg, ResultDev res, cudaStream_t st) {
  const Matrix& m = ctx->circ[ZK_CIRCUIT_PI];
  if (!(rg.flags & ZK_FLAG_WRAP) && rg.row_end + 1 > m.n_rows)
    return fail_msg(ctx, "pi rows [b,e) need row e resident (rotation +1) unless ZK_FLAG_WRAP");
  const u32 kk[5] = {0, 1, 2, 3, 4}, gk[3] = {0, 1, 2};
  IndexDev kec_ix, gas_ix;
  int rc;
  if ((rc = ensure_index(ctx, ZK_TABLE_KECCAK, kk, 5, st, &kec_ix))) return rc;
  if ((rc = ensure_index(ctx, ZK_TABLE_CALLDATA_GAS, gk, 3, st, &gas_ix))) return rc;
  if ((rc = mark_indexes_ready(ctx))) return rc;
  PiParams pp{fr_to_mont(ctx->chal[ZK_CHALLENGE_PI_KECCAK]), fr_to_mont(ctx->chal[ZK_CHALLENGE_PI_BYTE_BASE]),
              ctx->chal[ZK_PARAM_PI_CIRCUIT_LEN]};
  const u64 n = rg.row_end - rg.row_begin;
  if (is_canonical(m)) k_check_pi<L_CANON><<<grid_persistent(ctx, k_check_pi<L_CANON>, 256, n), 256, 0, st>>>(witness_dev(m), rg, kec_ix, gas_ix, pp, res);
  else k_check_pi<L_ANY><<<grid_persistent(ctx, k_check_pi<L_ANY>, 256, n), 256, 0, st>>>(witness_dev(m), rg, kec_ix, gas_ix, pp, res);
  ctx->launches++;
  CK(ctx, cudaGetLastError());
  return 0;
}

// the power table of the withdrawal circuit's RLC, rebuilt when ZK_CHALLENGE_KECCAK changed since the last build
static int ensure_wd_rpow(zk_ctx* ctx, cudaStream_t st) {
  const Fr& r = ctx->chal[ZK_CHALLENGE_KECCAK];
  if (ctx->wd_rpow && fr_eq(ctx->wd_rpow_r, r)) return 0;
  if (!ctx->wd_rpow) CK(ctx, cudaMalloc(&ctx->wd_rpow, WD_MAX_RLP * sizeof(Fr)));
  Fr host[WD_MAX_RLP];
  wd_rpow_table(r, host);
  CK(ctx, cudaMemcpyAsync(ctx->wd_rpow, host, sizeof(host), cudaMemcpyHostToDevice, st));
  CK(ctx, cudaStreamSynchronize(st));  // `host` goes out of scope
  ctx->wd_rpow_r = r;
  return 0;
}

static int wd_max(zk_ctx* ctx, u64* max) {
  const Fr& m = ctx->chal[ZK_PARAM_WITHDRAWAL_MAX];
  if (!fr_fits64(m) || m.l[0] >= 0xFFFFFFFFull) return fail_msg(ctx, "ZK_PARAM_WITHDRAWAL_MAX must be below 2^32 - 1");
  *max = m.l[0];
  return 0;
}

static int check_withdrawal(zk_ctx* ctx, const CheckRange& rg, ResultDev res, cudaStream_t st) {
  const Matrix& m = ctx->circ[ZK_CIRCUIT_WITHDRAWAL];
  u64 max;
  int rc;
  if ((rc = wd_max(ctx, &max))) return rc;
  const u64 gb = rg.row_base + rg.row_begin, ge = rg.row_base + rg.row_end;
  // global row 0 stands for rows[-1] when MAX == 0: the block lookup of an empty loop reads it
  if (ge > std::max<u64>(max, 1))
    return fail_msg(ctx, "withdrawal rows [b,e) reach past global row MAX - 1 (ZK_PARAM_WITHDRAWAL_MAX): later rows are not part of the circuit");
  if ((gb != 0 && rg.row_begin == 0) || (ge < max && rg.row_end + 1 > m.n_rows))
    return fail_msg(ctx, "withdrawal rows [b,e) need local row b-1 resident unless row_base + b == 0, and local row e resident "
                         "unless row_base + e == MAX (rotations -1,+1, no wrap)");
  const u32 kk[5] = {0, 1, 2, 3, 4}, k12[12] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11}, bk[3] = {0, 2, 3};
  IndexDev kec_ix, mpt_ix, blk_ix;
  if ((rc = ensure_index(ctx, ZK_TABLE_KECCAK, kk, 5, st, &kec_ix))) return rc;
  if ((rc = ensure_index(ctx, ZK_TABLE_MPT, k12, 12, st, &mpt_ix))) return rc;
  if ((rc = ensure_index(ctx, ZK_TABLE_BLOCK, bk, 3, st, &blk_ix))) return rc;
  if ((rc = ensure_wd_rpow(ctx, st))) return rc;
  if ((rc = mark_indexes_ready(ctx))) return rc;
  const u64 n = rg.row_end - rg.row_begin;
  if (is_canonical(m))
    k_check_withdrawal<L_CANON><<<grid_persistent(ctx, k_check_withdrawal<L_CANON>, 256, n), 256, 0, st>>>(witness_dev(m), rg, kec_ix, mpt_ix, blk_ix, ctx->wd_rpow, max, res);
  else
    k_check_withdrawal<L_ANY><<<grid_persistent(ctx, k_check_withdrawal<L_ANY>, 256, n), 256, 0, st>>>(witness_dev(m), rg, kec_ix, mpt_ix, blk_ix, ctx->wd_rpow, max, res);
  ctx->launches++;
  CK(ctx, cudaGetLastError());
  return 0;
}

// a resident matrix of canonical cells, n_rows x n_cols, that the library itself writes
static int own_canonical(zk_ctx* ctx, Matrix& m, u64 n_rows, u32 n_cols) {
  const size_t bytes = std::max<size_t>((size_t)n_rows * n_cols * 32, 32);
  if (m.borrowed) {
    m.dev = nullptr;
    m.borrowed = false;
    m.cap_bytes = 0;
  }
  if (bytes > m.cap_bytes) {
    if (m.dev) cudaFree(m.dev);
    m.dev = nullptr;
    CK(ctx, cudaMalloc(&m.dev, bytes));
    m.cap_bytes = bytes;
  }
  m.version++;
  m.n_rows = n_rows;
  m.n_cols = n_cols;
  m.flags_rows = 0;
  m.src_offsets = nullptr;
  m.narrow_mask = 0;
  layout_canonical(m.off, m.width, n_cols, n_rows);
  return 0;
}

extern "C" int zk_assign_withdrawal_circuit(zk_ctx* ctx, uint64_t n, const uint64_t* records, uint64_t max_withdrawals,
                                            void* stream) {
  CK(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  if (n > max_withdrawals) return fail_msg(ctx, "more withdrawals than max_withdrawals");
  if (max_withdrawals >= 0x7FFFFFFFull) return fail_msg(ctx, "max_withdrawals must be below 2^31 - 1");
  int rc;
  const size_t rec_bytes = std::max<size_t>((size_t)n * 20 * 8, 32);
  if (rec_bytes > ctx->wd_records_cap) {
    if (ctx->wd_records) cudaFree(ctx->wd_records);
    ctx->wd_records = nullptr;
    CK(ctx, cudaMalloc(&ctx->wd_records, rec_bytes));
    ctx->wd_records_cap = rec_bytes;
  }
  if (n) CK(ctx, cudaMemcpyAsync(ctx->wd_records, records, (size_t)n * 20 * 8, cudaMemcpyHostToDevice, st));
  Matrix& rows = ctx->circ[ZK_CIRCUIT_WITHDRAWAL];
  Matrix& kec = ctx->tab[ZK_TABLE_KECCAK];
  if ((rc = own_canonical(ctx, rows, max_withdrawals, WD_COLS))) return rc;
  if ((rc = own_canonical(ctx, kec, n + 1, 5))) return rc;
  if ((rc = ensure_wd_rpow(ctx, st))) return rc;
  if (max_withdrawals == 0) {  // no row to write: the keccak table is the all-zero row alone
    CK(ctx, cudaMemsetAsync(kec.dev, 0, 5 * 32, st));
    return 0;
  }
  const unsigned grid = (unsigned)std::min<u64>((max_withdrawals + WD_ASSIGN_THREADS - 1) / WD_ASSIGN_THREADS, (u64)ctx->sm_count * 16);
  k_assign_withdrawal<<<grid, WD_ASSIGN_THREADS, 0, st>>>(ctx->wd_records, n, max_withdrawals, ctx->wd_rpow, rows.dev, kec.dev);
  ctx->launches++;
  CK(ctx, cudaGetLastError());
  return 0;
}

static int check_state(zk_ctx* ctx, const CheckRange& rg, ResultDev res, cudaStream_t st) {
  const Matrix& m = ctx->circ[ZK_CIRCUIT_STATE];
  if (!(rg.flags & ZK_FLAG_WRAP) && (rg.row_begin == 0 || rg.row_end + 1 > m.n_rows))
    return fail_msg(ctx, "state rows [b,e) need rows b-1 and e resident (rotations -1,+1) unless ZK_FLAG_WRAP");
  const u32 k12[12] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11};
  IndexDev mpt;
  int rc;
  if ((rc = ensure_index(ctx, ZK_TABLE_MPT, k12, 12, st, &mpt))) return rc;
  if ((rc = mark_indexes_ready(ctx))) return rc;
  const u64 n = rg.row_end - rg.row_begin;
  // fold pass over every resident row (halos included), then the gate program
  if (m.n_rows * sizeof(StateFold) > ctx->state_fold_cap) {
    if (ctx->state_fold) cudaFree(ctx->state_fold);
    ctx->state_fold = nullptr;
    CK(ctx, cudaMalloc(&ctx->state_fold, m.n_rows * sizeof(StateFold)));
    ctx->state_fold_cap = m.n_rows * sizeof(StateFold);
  }
  StateFold* fold = (StateFold*)ctx->state_fold;
  const WitnessDev wd = witness_dev(m);
  if (is_canonical(m)) {
    k_state_fold<L_CANON><<<grid_persistent(ctx, k_state_fold<L_CANON>, 256, m.n_rows), 256, 0, st>>>(wd, fold);
    k_check_state<L_CANON><<<grid_persistent(ctx, k_check_state<L_CANON>, 128, n), 128, 0, st>>>(wd, rg, mpt, res, fold);
  } else {
    k_state_fold<L_ANY><<<grid_persistent(ctx, k_state_fold<L_ANY>, 256, m.n_rows), 256, 0, st>>>(wd, fold);
    k_check_state<L_ANY><<<grid_persistent(ctx, k_check_state<L_ANY>, 128, n), 128, 0, st>>>(wd, rg, mpt, res, fold);
  }
  ctx->launches += 2;
  CK(ctx, cudaGetLastError());
  return 0;
}

static int check_copy(zk_ctx* ctx, const CheckRange& rg, ResultDev res, cudaStream_t st) {
  const Matrix& m = ctx->circ[ZK_CIRCUIT_COPY];
  if (!(rg.flags & ZK_FLAG_WRAP) && rg.row_end + 2 > m.n_rows)
    return fail_msg(ctx, "copy rows [b,e) need rows e and e+1 resident (rotations +1,+2) unless ZK_FLAG_WRAP");
  const u32 k5[5] = {0, 1, 2, 3, 4}, k3[3] = {0, 1, 2};
  CopyTables t;
  int rc;
  if ((rc = ensure_index(ctx, ZK_TABLE_RW, k5, 5, st, &t.rw, ZK_POS_DENSE))) return rc;
  if ((rc = ensure_index(ctx, ZK_TABLE_BYTECODE, k5, 5, st, &t.bytecode, ZK_POS_RUNS))) return rc;
  if ((rc = ensure_index(ctx, ZK_TABLE_TX, k3, 3, st, &t.tx))) return rc;
  if ((rc = mark_indexes_ready(ctx))) return rc;
  const u64 n = rg.row_end - rg.row_begin;
  const Fr r_mont = fr_to_mont(ctx->chal[ZK_CHALLENGE_KECCAK]);
  // deferred-warp list of the small / general split (copy.cu): one u32 per 32 rows + the counter
  const size_t need = (n / 32 + 2) * sizeof(u32);
  if (need > ctx->copy_slow_cap) {
    if (ctx->copy_slow) cudaFree(ctx->copy_slow);
    ctx->copy_slow = nullptr;
    CK(ctx, cudaMalloc(&ctx->copy_slow, need));
    ctx->copy_slow_cap = need;
  }
  CK(ctx, cudaMemsetAsync(ctx->copy_slow, 0, sizeof(u32), st));
  const CopySlowList slow{ctx->copy_slow, ctx->copy_slow + 1};
  const unsigned g_general = (unsigned)std::min<u64>((n / 32 + 3) / 4 + 1, (u64)ctx->sm_count * 2);
  if (is_canonical(m)) {
    k_check_copy_small<L_CANON><<<grid_persistent(ctx, k_check_copy_small<L_CANON>, 128, n), 128, 0, st>>>(witness_dev(m), rg, t, r_mont, res, slow);
    k_check_copy_general<L_CANON><<<g_general, 128, 0, st>>>(witness_dev(m), rg, t, r_mont, res, slow);
  } else {
    k_check_copy_small<L_ANY><<<grid_persistent(ctx, k_check_copy_small<L_ANY>, 128, n), 128, 0, st>>>(witness_dev(m), rg, t, r_mont, res, slow);
    k_check_copy_general<L_ANY><<<g_general, 128, 0, st>>>(witness_dev(m), rg, t, r_mont, res, slow);
  }
  ctx->launches += 2;
  CK(ctx, cudaGetLastError());
  return 0;
}

static int ensure_aux_stream(zk_ctx* ctx) {
  if (!ctx->evm_aux) {
    CK(ctx, cudaStreamCreateWithFlags(&ctx->evm_aux, cudaStreamNonBlocking));
    CK(ctx, cudaEventCreateWithFlags(&ctx->evm_fork_ev, cudaEventDisableTiming));
    CK(ctx, cudaEventCreateWithFlags(&ctx->evm_join_ev, cudaEventDisableTiming));
    CK(ctx, cudaEventCreateWithFlags(&ctx->evm_index_join_ev, cudaEventDisableTiming));
  }
  return 0;
}

// the narrow instances of the hot EVM kernels (evm.cu StepCtx::narrow) apply when the resident step matrix, rw table
// and bytecode table have these storage properties (every packer / the from-code upload produces them on real traces)
static bool evm_narrow(const zk_ctx* ctx) {
  const Matrix& sm = ctx->circ[ZK_CIRCUIT_EVM];
  const Matrix& rw = ctx->tab[ZK_TABLE_RW];
  const Matrix& bt = ctx->tab[ZK_TABLE_BYTECODE];
  const u64 step_need = 0x1FFFull & ~((1ull << 5) | (1ull << 6));  // all 13 step cells but code_hash lo / hi
  if ((sm.narrow_mask & step_need) != step_need) return false;
  if ((rw.narrow_mask & 0x1Full) != 0x1Full) return false;  // rw_counter, rw, tag, id, address
  static const unsigned char kW[6] = {16, 16, 1, 4, 1, 4};
  for (int c = 0; c < 6; c++)
    if (bt.width[c] != kW[c]) return false;
  return bt.n_cols == 6;
}

static int check_evm(zk_ctx* ctx, const CheckRange& rg, ResultDev res, cudaStream_t st) {
  const Matrix& m = ctx->circ[ZK_CIRCUIT_EVM];
  if (rg.row_end + 1 > m.n_rows) return fail_msg(ctx, "EVM steps [b,e) need step e resident (rotation +1)");
  const u32 k5[5] = {0, 1, 2, 3, 4}, k4[4] = {0, 1, 2, 3};
  EvmTables t;
  int rc;
  // The bytecode and rw indexes: one k_pos_prep for both, the bytecode verify (its heads index serves classify's
  // opcode peek), then the rw verify — on the auxiliary stream underneath classify + scatter, which never read the rw
  // table.  Their hash parts wait for the flags, which the host reads back with the histogram.
  Index* ixs[2];  // bytecode, rw
  if ((rc = find_index(ctx, ZK_TABLE_BYTECODE, k5, 5, ZK_POS_RUNS, st, &ixs[0]))) return rc;
  if ((rc = find_index(ctx, ZK_TABLE_RW, k5, 5, ZK_POS_DENSE, st, &ixs[1]))) return rc;
  bool rebuild[2];
  Index* prep[2];
  u32 n_prep = 0;
  for (int e = 0; e < 2; e++) {
    rebuild[e] = !index_current(ctx, ixs[e]);
    if (!rebuild[e]) ixs[e]->dev.tab = table_dev(ctx, ixs[e]->table_id);  // flags may have been (re)uploaded
    else if ((rc = describe_index(ctx, ixs[e]))) return rc;
    if (rebuild[e] && ixs[e]->dev.pos_ok) prep[n_prep++] = ixs[e];
  }
  if ((rc = launch_pos_prep(ctx, prep, n_prep, st))) return rc;
  if (rebuild[0]) {
    if (ixs[0]->dev.pos_ok && (rc = launch_pos_verify(ctx, ixs[0], st))) return rc;
    if ((rc = finish_index(ctx, ixs[0], st, true))) return rc;
  }
  t.bytecode = ixs[0]->dev;
  t.rw = ixs[1]->dev;
  if ((rc = ensure_index(ctx, ZK_TABLE_FIXED, k4, 4, st, &t.fixed))) return rc;
  {
    const u32 ck[11] = {1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 12}, kk[3] = {0, 1, 2};
    if ((rc = ensure_index(ctx, ZK_TABLE_COPY, ck, 11, st, &t.copy))) return rc;
    if ((rc = ensure_index(ctx, ZK_TABLE_KECCAK, kk, 3, st, &t.keccak))) return rc;
    const u32 tk[3] = {0, 1, 2}, bk[2] = {0, 1};
    if ((rc = ensure_index(ctx, ZK_TABLE_TX, tk, 3, st, &t.tx))) return rc;
    if ((rc = ensure_index(ctx, ZK_TABLE_BLOCK, bk, 2, st, &t.block))) return rc;
    const u32 ek[9] = {0, 1, 2, 3, 4, 5, 6, 7, 8};
    if ((rc = ensure_index(ctx, ZK_TABLE_EXP, ek, 9, st, &t.exp))) return rc;
    const u32 ak[1] = {0};
    if ((rc = ensure_index(ctx, ZK_TABLE_STEP_AUX, ak, 1, st, &t.aux))) return rc;
  }
  if (!ctx->resp_bitmap) CK(ctx, cudaMalloc(&ctx->resp_bitmap, ZK_RESP_BITMAP_WORDS * sizeof(u32)));
  if (ctx->resp_bitmap_version != ctx->tab[ZK_TABLE_FIXED].version) {
    CK(ctx, cudaMemsetAsync(ctx->resp_bitmap, 0, ZK_RESP_BITMAP_WORDS * sizeof(u32), st));
    if (t.fixed.tab.n_rows) {
      k_fixed_resp_bitmap<<<(unsigned)((t.fixed.tab.n_rows + 255) / 256), 256, 0, st>>>(t.fixed.tab, ctx->resp_bitmap);
      ctx->launches++;
    }
    ctx->resp_bitmap_version = ctx->tab[ZK_TABLE_FIXED].version;
  }
  t.resp_bitmap = ctx->resp_bitmap;
  t.wd = table_dev(ctx, ZK_TABLE_WITHDRAWAL);
  t.stats = nullptr;
  if (!ctx->evm_hist_host) {
    CK(ctx, cudaHostAlloc(&ctx->evm_hist_host, (ZK_EVM_NB + 5) * sizeof(u32), cudaHostAllocDefault));
    CK(ctx, cudaEventCreateWithFlags(&ctx->evm_hist_ev, cudaEventDisableTiming));
  }
  // read-back of the two flags: [0] bytecode, [2] rw (0 for an empty table, whose flag is never initialised)
  u32* flags_host = ctx->evm_hist_host + ZK_EVM_NB + 1;
  for (int e = 0; e < 4; e++) flags_host[e] = 0;
  auto copy_flags = [&](cudaStream_t s_) -> int {
    for (int e = 0; e < 2; e++)
      if (ixs[e]->dev.pos_ok) CK(ctx, cudaMemcpyAsync(flags_host + 2 * e, ixs[e]->pos_flag, 2 * sizeof(u32), cudaMemcpyDeviceToHost, s_));
    return 0;
  };
  if (ctx->evm_index_overlap < 0) {
    const char* e_ = getenv("ZKCHECK_INDEX_OVERLAP");
    ctx->evm_index_overlap = (e_ && e_[0] == '0') ? 0 : 1;
  }
  const bool rw_verify = rebuild[1] && ixs[1]->dev.pos_ok;
  const bool index_forked = rw_verify && ctx->evm_index_overlap;
  if (index_forked) {  // the fork point; the verify itself is enqueued after classify, which the host launches first
    if ((rc = ensure_aux_stream(ctx))) return rc;
    CK(ctx, cudaEventRecord(ctx->evm_fork_ev, st));
  } else if (rw_verify) {
    if ((rc = launch_pos_verify(ctx, ixs[1], st))) return rc;
  }
  if (rebuild[1] && (rc = finish_index(ctx, ixs[1], st, true))) return rc;
  if ((rc = mark_indexes_ready(ctx))) return rc;
  const u64 n = rg.row_end - rg.row_begin;
  // counting sort of the steps by execution state (k_evm_classify + k_evm_scatter), then one kernel
  // per non-empty gate-program group
  auto up256 = [](size_t x) { return (x + 255) / 256 * 256; };
  if (n > ctx->evm_sort_cap) {
    if (ctx->evm_sort) cudaFree(ctx->evm_sort);
    ctx->evm_sort = nullptr;
    CK(ctx, cudaMalloc(&ctx->evm_sort, up256(n) + up256(n * 4) + (3 * ZK_EVM_NB + 2) * sizeof(u32)));
    ctx->evm_sort_cap = n;
  }
  EvmSort so;
  so.bucket = ctx->evm_sort;
  so.sorted = (u32*)(ctx->evm_sort + up256(ctx->evm_sort_cap));
  so.hist = (u32*)(ctx->evm_sort + up256(ctx->evm_sort_cap) + up256(ctx->evm_sort_cap * 4));
  so.cursor = so.hist + ZK_EVM_NB + 1;
  so.offs = so.cursor + ZK_EVM_NB;
  CK(ctx, cudaMemsetAsync(so.hist, 0, (2 * ZK_EVM_NB + 1) * sizeof(u32), st));
  const WitnessDev wd = witness_dev(m);
  const unsigned sort_grid = (unsigned)((n + 1023) / 1024);
  // the narrow instance needs 40 registers: blocks of ZK_CLASSIFY_THREADS = 512 keep 48 warps resident per SM instead of 32
#ifndef ZK_CLASSIFY_THREADS
#define ZK_CLASSIFY_THREADS 512
#endif
  if (evm_narrow(ctx)) k_evm_classify<1><<<(unsigned)((n + ZK_CLASSIFY_THREADS - 1) / ZK_CLASSIFY_THREADS), ZK_CLASSIFY_THREADS, 0, st>>>(wd, rg, t, res, so);
  else k_evm_classify<0><<<sort_grid, 1024, 0, st>>>(wd, rg, t, res, so);
  {
    cudaError_t e_ = cudaGetLastError();
    if (e_ != cudaSuccess) return fail_msg(ctx, std::string("launch of k_evm_classify: ") + cudaGetErrorString(e_));
  }
  if (index_forked) {
    CK(ctx, cudaStreamWaitEvent(ctx->evm_aux, ctx->evm_fork_ev, 0));
    if ((rc = launch_pos_verify(ctx, ixs[1], ctx->evm_aux))) return rc;
    if ((rc = copy_flags(ctx->evm_aux))) return rc;
    CK(ctx, cudaEventRecord(ctx->evm_index_join_ev, ctx->evm_aux));
  }
  CK(ctx, cudaMemcpyAsync(ctx->evm_hist_host, so.hist, ZK_EVM_NB * sizeof(u32), cudaMemcpyDeviceToHost, st));
  if (!index_forked && (rc = copy_flags(st))) return rc;
  CK(ctx, cudaEventRecord(ctx->evm_hist_ev, st));
  k_evm_scatter<<<sort_grid, 1024, 0, st>>>(so, (u32)n);
  ctx->launches += 2;
  {
    cudaError_t e_ = cudaGetLastError();
    if (e_ != cudaSuccess) return fail_msg(ctx, std::string("launch of k_evm_scatter: ") + cudaGetErrorString(e_));
  }
  // the join: nothing after this point on `st` runs before the rw verify is done
  if (index_forked) CK(ctx, cudaStreamWaitEvent(st, ctx->evm_index_join_ev, 0));
  // the histogram decides which groups run and how large their grids are, the flags which kernel forms run and which
  // hash parts are built; the device keeps working on the scatter meanwhile
  CK(ctx, cudaEventSynchronize(ctx->evm_hist_ev));
  if (index_forked) CK(ctx, cudaEventSynchronize(ctx->evm_index_join_ev));
  const u32* hist = ctx->evm_hist_host;
  const bool bc_pos = flags_host[0] != 0, rw_pos = flags_host[2] != 0;
  const bool pos = bc_pos && rw_pos;  // both_positional (evm.cu)
  if ((rc = resolve_hash(ctx, ixs[0], bc_pos, st))) return rc;
  if ((rc = resolve_hash(ctx, ixs[1], rw_pos, st))) return rc;
  u64 group_n[KG_COUNT] = {0};
  for (int b = 0; b < ZK_EVM_NB; b++) {
    const int g = es_group(b);
    if (g >= 0) group_n[g] += hist[b];
  }
  // transaction-level steps (BeginTx / EndTx / EndBlock) look rw rows up by other column subsets: a dense rw
  // table serves them by position, otherwise through an index on rw_counter alone, built only now that such
  // steps are known to exist; EndBlock also needs the table-derived constants
  const u64 n_tx_level = (u64)hist[ZK_ES_BeginTx] + hist[ZK_ES_EndTx] + hist[ZK_ES_EndBlock] + hist[ZK_ES_SELFBALANCE] +
                         hist[ZK_ES_BALANCE] + hist[ZK_ES_EXTCODEHASH] + hist[ZK_ES_EXTCODESIZE] + hist[ZK_ES_ErrorOutOfGasAccountAccess] +
                         hist[ZK_ES_EXTCODECOPY] + hist[ZK_ES_ErrorOutOfGasMemoryCopy] + hist[ZK_ES_SLOAD] + hist[ZK_ES_SSTORE] +
                         hist[ZK_ES_CALLDATALOAD] + hist[ZK_ES_LOG] + hist[ZK_ES_ErrorWriteProtection] + hist[ZK_ES_ErrorMaxCodeSizeExceeded] +
                         hist[ZK_ES_ErrorOutOfGasCodeStore] + hist[ZK_ES_ErrorInvalidCreationCode] + hist[ZK_ES_RETURN] + hist[ZK_ES_ErrorOutOfGasCall] + hist[ZK_ES_CALL_OP] +
                         hist[ZK_ES_CREATE] + hist[ZK_ES_CREATE2] + hist[ZK_ES_ErrorOutOfGasSloadSstore] + hist[ZK_ES_ErrorOutOfGasCREATE] +
                         hist[ZK_ES_ErrorOutOfGasPrecompile] + hist[ZK_ES_ErrorGasUintOverflow];
  if (hist[ZK_ES_ErrorInvalidJump] && !pos) {  // bytecode_lookup_pair: the index without is_code
    const u32 k4b[4] = {0, 1, 2, 3};
    if ((rc = ensure_index(ctx, ZK_TABLE_BYTECODE, k4b, 4, st, &t.bytecode4))) return rc;
  }
  if (n_tx_level) {
    const u32 k1[1] = {0};
    if (!pos && (rc = ensure_index(ctx, ZK_TABLE_RW, k1, 1, st, &t.rw_rwc))) return rc;
    if (hist[ZK_ES_EndBlock]) {
      if (!ctx->block_stats) CK(ctx, cudaMalloc(&ctx->block_stats, sizeof(BlockStats)));
      CK(ctx, cudaMemsetAsync(ctx->block_stats, 0, sizeof(BlockStats), st));
      const u64 rows = std::max<u64>(std::max<u64>(t.tx.tab.n_rows, t.wd.n_rows), pos ? 1 : t.rw.tab.n_rows);
      k_evm_block_stats<<<(unsigned)std::max<u64>(1, std::min<u64>((rows + 255) / 256, (u64)ctx->sm_count * 8)), 256, 0, st>>>(t, ctx->block_stats);
      ctx->launches++;
      t.stats = ctx->block_stats;
    }
  }
  // persistent grids: at most the number of blocks the device keeps resident (occupancy x SMs), each
  // thread walks its bucket with a grid stride
  auto grid_for = [&](int slot, const void* kernel, u64 work_items, unsigned per_block) -> unsigned {
    if (!ctx->evm_occ[slot]) {
      int occ = 0;
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, 128, 0) != cudaSuccess || occ < 1) occ = 1;
      ctx->evm_occ[slot] = occ;
    }
    const u64 want = (work_items + per_block - 1) / per_block;
    return (unsigned)std::max<u64>(1, std::min<u64>(want, (u64)ctx->evm_occ[slot] * ctx->sm_count));
  };
#define ZK_LAUNCH_GROUP(slot, kernel, items, per_block) ZK_LAUNCH_GROUP_ON(st, slot, kernel, items, per_block)
#define ZK_LAUNCH_GROUP_ON(stream_, slot, kernel, items, per_block)                            \
  do {                                                                                         \
    kernel<<<grid_for(slot, (const void*)kernel, items, per_block), 128, 0, stream_>>>(wd, rg, t, res, so); \
    ctx->launches++;                                                                           \
    {                                                                                          \
      cudaError_t e_ = cudaGetLastError();                                                     \
      if (e_ != cudaSuccess) return fail_msg(ctx, std::string("launch of " #kernel ": ") + cudaGetErrorString(e_)); \
    }                                                                                          \
  } while (0)
  // narrow instances: positional tables AND every step column but the code hash, the rw table's key columns narrow
  // (<= 8 bytes per row, Matrix::narrow_mask) AND the bytecode table in the layout k_bytecode_table_expand writes
  const bool narrow = pos && evm_narrow(ctx);
  // the transaction-level group first, on the auxiliary stream: its blocks take their places before the hot kernels'
  // persistent grids fill the device, and its long per-thread chains run underneath them
  bool tx_forked = false;
  if (group_n[KG_TX]) {
    if (ctx->evm_tx_overlap < 0) {
      const char* e_ = getenv("ZKCHECK_TX_OVERLAP");
      ctx->evm_tx_overlap = (e_ && e_[0] == '0') ? 0 : 1;
    }
    if (ctx->evm_tx_overlap) {
      if ((rc = ensure_aux_stream(ctx))) return rc;
      CK(ctx, cudaEventRecord(ctx->evm_fork_ev, st));
      CK(ctx, cudaStreamWaitEvent(ctx->evm_aux, ctx->evm_fork_ev, 0));
      ZK_LAUNCH_GROUP_ON(ctx->evm_aux, 12, k_evm_group<KG_TX>, group_n[KG_TX], 128);
      CK(ctx, cudaEventRecord(ctx->evm_join_ev, ctx->evm_aux));
      tx_forked = true;
    }
  }
  if (group_n[KG_PUSH]) {
    if (narrow) ZK_LAUNCH_GROUP(13, k_evm_push_pos<1>, group_n[KG_PUSH], 128);
    else if (pos) ZK_LAUNCH_GROUP(0, k_evm_push_pos<0>, group_n[KG_PUSH], 128);
    else ZK_LAUNCH_GROUP(1, k_evm_push_hash, group_n[KG_PUSH], 8);  // half a warp per step
  }
  if (group_n[KG_MUL]) {
    if (narrow) ZK_LAUNCH_GROUP(14, (k_evm_gadget<KG_MUL, 2>), group_n[KG_MUL], 128);
    else if (pos) ZK_LAUNCH_GROUP(2, (k_evm_gadget<KG_MUL, 1>), group_n[KG_MUL], 128);
    else ZK_LAUNCH_GROUP(3, (k_evm_gadget<KG_MUL, 0>), group_n[KG_MUL], 128);
  }
  if (group_n[KG_ADD]) {
    if (narrow) ZK_LAUNCH_GROUP(15, (k_evm_gadget<KG_ADD, 2>), group_n[KG_ADD], 128);
    else if (pos) ZK_LAUNCH_GROUP(4, (k_evm_gadget<KG_ADD, 1>), group_n[KG_ADD], 128);
    else ZK_LAUNCH_GROUP(5, (k_evm_gadget<KG_ADD, 0>), group_n[KG_ADD], 128);
  }
  if (group_n[KG_POP]) {
    if (narrow) ZK_LAUNCH_GROUP(16, (k_evm_gadget<KG_POP, 2>), group_n[KG_POP], 128);
    else if (pos) ZK_LAUNCH_GROUP(6, (k_evm_gadget<KG_POP, 1>), group_n[KG_POP], 128);
    else ZK_LAUNCH_GROUP(7, (k_evm_gadget<KG_POP, 0>), group_n[KG_POP], 128);
  }
  if (group_n[KG_SIMPLE]) ZK_LAUNCH_GROUP(8, k_evm_group<KG_SIMPLE>, group_n[KG_SIMPLE], 128);
  if (group_n[KG_BYTES32]) ZK_LAUNCH_GROUP(9, k_evm_group<KG_BYTES32>, group_n[KG_BYTES32], 128);
  if (group_n[KG_COPY]) ZK_LAUNCH_GROUP(10, k_evm_group<KG_COPY>, group_n[KG_COPY], 128);
  if (group_n[KG_WIDE]) ZK_LAUNCH_GROUP(11, k_evm_group<KG_WIDE>, group_n[KG_WIDE], 128);
  if (group_n[KG_TX] && !tx_forked) ZK_LAUNCH_GROUP(12, k_evm_group<KG_TX>, group_n[KG_TX], 128);
  if (group_n[KG_ARITH]) ZK_LAUNCH_GROUP(17, k_evm_group<KG_ARITH>, group_n[KG_ARITH], 128);
  if (tx_forked) CK(ctx, cudaStreamWaitEvent(st, ctx->evm_join_ev, 0));
#undef ZK_LAUNCH_GROUP
#undef ZK_LAUNCH_GROUP_ON
  CK(ctx, cudaGetLastError());
  return 0;
}

extern "C" int zk_check_async(zk_ctx* ctx, int circuit_id, uint64_t row_begin, uint64_t row_end,
                              uint64_t row_base, uint32_t flags, void* stream) {
  if (circuit_id < 0 || circuit_id >= ZK_N_CIRCUITS) return fail_msg(ctx, "bad circuit id");
  CK(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  const Matrix& m = ctx->circ[circuit_id];
  if (!m.dev && m.n_rows) return fail_msg(ctx, "no witness uploaded for circuit");
  if (row_begin > row_end || row_end > m.n_rows) return fail_msg(ctx, "row range outside the resident matrix");
  // reported rows are row_base + i (mod 2^64: a shard whose first resident row is a halo passes row_base = -1)
  if (row_base + row_begin + (row_end - row_begin) >= 0xFFFFFFFFull || row_base + row_begin >= 0xFFFFFFFFull)
    return fail_msg(ctx, "reported rows row_base + [row_begin, row_end) must stay below 2^32 - 1 (first_fail holds uint32 rows, 0xFFFFFFFF = pass)");
  ResultDev res;
  int rc = ensure_result(ctx, circuit_id, &res, st);
  if (rc) return rc;
  if (row_begin == row_end) return 0;
  CheckRange rg{row_begin, row_end, row_base, flags};
  {  // an error left behind by an earlier call must not be blamed on this check's launches
    cudaError_t stale = cudaGetLastError();
    if (stale != cudaSuccess) return fail_msg(ctx, std::string("CUDA error pending before the check: ") + cudaGetErrorString(stale));
  }
  ctx->ev_mid_stream = st;
  if (ctx->timing) CK(ctx, cudaEventRecord(ctx->ev[0], st));
  switch (circuit_id) {
    case ZK_CIRCUIT_BYTECODE: rc = check_bytecode(ctx, rg, res, st); break;
    case ZK_CIRCUIT_EVM: rc = check_evm(ctx, rg, res, st); break;
    case ZK_CIRCUIT_COPY: rc = check_copy(ctx, rg, res, st); break;
    case ZK_CIRCUIT_STATE: rc = check_state(ctx, rg, res, st); break;
    case ZK_CIRCUIT_EXP: rc = check_exp(ctx, rg, res, st); break;
    case ZK_CIRCUIT_TX: rc = check_tx(ctx, rg, res, st); break;
    case ZK_CIRCUIT_SIG: rc = check_tx(ctx, rg, res, st, true); break;
    case ZK_CIRCUIT_PI: rc = check_pi(ctx, rg, res, st); break;
    case ZK_CIRCUIT_WITHDRAWAL: rc = check_withdrawal(ctx, rg, res, st); break;
    default: return fail_msg(ctx, "circuit has no gate program in this build");
  }
  if (rc) return rc;
  if (ctx->timing) CK(ctx, cudaEventRecord(ctx->ev[2], st));
  return 0;
}

// called by the per-circuit dispatchers between the index builds and the circuit kernel
static int mark_indexes_ready(zk_ctx* ctx) {
  if (ctx->timing) CK(ctx, cudaEventRecord(ctx->ev[1], ctx->ev_mid_stream));
  return 0;
}

extern "C" int zk_enable_timing(zk_ctx* ctx, int on) {
  CK(ctx, cudaSetDevice(ctx->device));
  if (on && !ctx->ev[0])
    for (auto& e : ctx->ev) CK(ctx, cudaEventCreate(&e));
  ctx->timing = on != 0;
  return 0;
}
extern "C" int zk_last_timing(zk_ctx* ctx, float* index_ms, float* check_ms) {
  if (!ctx->timing) return fail_msg(ctx, "timing not enabled");
  CK(ctx, cudaEventSynchronize(ctx->ev[2]));
  if (index_ms) CK(ctx, cudaEventElapsedTime(index_ms, ctx->ev[0], ctx->ev[1]));
  if (check_ms) CK(ctx, cudaEventElapsedTime(check_ms, ctx->ev[1], ctx->ev[2]));
  return 0;
}

extern "C" int zk_result_device(zk_ctx* ctx, int circuit_id, uint32_t** ff, uint64_t** fc) {
  if (circuit_id < 0 || circuit_id >= ZK_N_CIRCUITS) return fail_msg(ctx, "bad circuit id");
  ResultBuf& r = ctx->res[circuit_id];
  if (!r.first_fail) return fail_msg(ctx, "no result yet");
  if (ff) *ff = r.first_fail;
  if (fc) *fc = (uint64_t*)r.fail_count;
  return 0;
}

extern "C" int zk_fetch_result(zk_ctx* ctx, int circuit_id, uint32_t* first_fail,
                               uint64_t* fail_count, void* stream) {
  if (circuit_id < 0 || circuit_id >= ZK_N_CIRCUITS) return fail_msg(ctx, "bad circuit id");
  CK(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  ResultBuf& r = ctx->res[circuit_id];
  if (!r.first_fail) return fail_msg(ctx, "no result yet");
  if (first_fail)
    CK(ctx, cudaMemcpyAsync(first_fail, r.first_fail, (size_t)r.n * 4, cudaMemcpyDeviceToHost, st));
  if (fail_count)
    CK(ctx, cudaMemcpyAsync(fail_count, r.fail_count, (size_t)r.n * 8, cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaStreamSynchronize(st));
  return 0;
}

extern "C" int zk_check(zk_ctx* ctx, int circuit_id, uint64_t row_begin, uint64_t row_end,
                        uint64_t row_base, uint32_t flags, uint32_t* first_fail,
                        uint64_t* fail_count, void* stream) {
  int rc = zk_check_async(ctx, circuit_id, row_begin, row_end, row_base, flags, stream);
  if (rc) return rc;
  return zk_fetch_result(ctx, circuit_id, first_fail, fail_count, stream);
}

// ------------------------------------------------------------------ multi-GPU
// NCCL is bound at run time (dlopen) so that libzkcheck.so has no link-time dependency on a
// particular libnccl; a process that already loaded one (e.g. through torch) gets that same library.
struct Id128 {  // ncclUniqueId: 128 opaque bytes, passed by value
  char b[128];
};
struct NcclApi {
  int (*get_unique_id)(void*) = nullptr;
  int (*comm_init_rank)(void**, int, Id128, int) = nullptr;
  int (*comm_destroy)(void*) = nullptr;
  int (*comm_count)(void*, int*) = nullptr;
  int (*all_gather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
  bool ok = false;
};
static NcclApi g_nccl;
static int nccl_bind(zk_ctx* ctx) {
  if (g_nccl.ok) return 0;
  void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!h) return fail_msg(ctx, std::string("cannot load NCCL: ") + dlerror());
  g_nccl.get_unique_id = (int (*)(void*))dlsym(h, "ncclGetUniqueId");
  g_nccl.comm_init_rank = (int (*)(void**, int, Id128, int))dlsym(h, "ncclCommInitRank");
  g_nccl.comm_destroy = (int (*)(void*))dlsym(h, "ncclCommDestroy");
  g_nccl.comm_count = (int (*)(void*, int*))dlsym(h, "ncclCommCount");
  g_nccl.all_gather = (int (*)(const void*, void*, size_t, int, void*, cudaStream_t))dlsym(h, "ncclAllGather");
  if (!g_nccl.get_unique_id || !g_nccl.comm_init_rank || !g_nccl.comm_destroy || !g_nccl.comm_count || !g_nccl.all_gather)
    return fail_msg(ctx, "NCCL symbols not found");
  g_nccl.ok = true;
  return 0;
}
extern "C" int zk_nccl_unique_id(zk_ctx* ctx, uint8_t id[128]) {
  int rc = nccl_bind(ctx);
  if (rc) return rc;
  if (g_nccl.get_unique_id(id)) return fail_msg(ctx, "ncclGetUniqueId failed");
  return 0;
}
extern "C" int zk_nccl_comm_init(zk_ctx* ctx, int world, int rank, const uint8_t id[128], void** comm) {
  int rc = nccl_bind(ctx);
  if (rc) return rc;
  CK(ctx, cudaSetDevice(ctx->device));
  Id128 u;
  memcpy(u.b, id, 128);
  if (g_nccl.comm_init_rank(comm, world, u, rank)) return fail_msg(ctx, "ncclCommInitRank failed");
  return 0;
}
extern "C" int zk_nccl_comm_destroy(zk_ctx* ctx, void* comm) {
  int rc = nccl_bind(ctx);
  if (rc) return rc;
  return g_nccl.comm_destroy(comm) ? fail_msg(ctx, "ncclCommDestroy failed") : 0;
}

// after the all-gather: first_fail = MIN over ranks, fail_count = SUM over ranks, in place
__global__ void k_reduce_results(const unsigned char* gathered, size_t rank_bytes, size_t count_off, int world, int n,
                                 u32* first_fail, u64* fail_count) {
  const int id = blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= n) return;
  u32 mn = 0xFFFFFFFFu;
  u64 sum = 0;
  for (int r = 0; r < world; r++) {
    const unsigned char* p = gathered + (size_t)r * rank_bytes;
    mn = min(mn, ((const u32*)p)[id]);
    sum += ((const u64*)(p + count_off))[id];
  }
  first_fail[id] = mn;
  fail_count[id] = sum;
}

// ONE collective: every rank's result vector (first_fail | fail_count, a few KB) is all-gathered, then
// a one-block kernel folds the copies (MIN / SUM do not share a reduction op, an all-reduce would
// need two rounds)
extern "C" int zk_allreduce_results(zk_ctx* ctx, int circuit_id, void* nccl_comm, void* stream) {
  if (circuit_id < 0 || circuit_id >= ZK_N_CIRCUITS) return fail_msg(ctx, "bad circuit id");
  ResultBuf& r = ctx->res[circuit_id];
  if (!r.first_fail) return fail_msg(ctx, "no result yet");
  int rc = nccl_bind(ctx);
  if (rc) return rc;
  CK(ctx, cudaSetDevice(ctx->device));
  int world = 0;
  if (g_nccl.comm_count(nccl_comm, &world) || world < 1) return fail_msg(ctx, "ncclCommCount failed");
  const size_t count_off = (size_t)((const char*)r.fail_count - (const char*)r.first_fail);
  const size_t rank_bytes = count_off + (size_t)r.n * 8;
  if (ctx->gather_cap < rank_bytes * world) {
    if (ctx->gather) cudaFree(ctx->gather);
    ctx->gather = nullptr;
    CK(ctx, cudaMalloc(&ctx->gather, rank_bytes * world));
    ctx->gather_cap = rank_bytes * world;
  }
  cudaStream_t st = (cudaStream_t)stream;
  // ncclChar = 0 (nccl.h)
  if (g_nccl.all_gather(r.first_fail, ctx->gather, rank_bytes, 0, nccl_comm, st)) return fail_msg(ctx, "ncclAllGather failed");
  k_reduce_results<<<(r.n + 255) / 256, 256, 0, st>>>(ctx->gather, rank_bytes, count_off, world, r.n, r.first_fail, r.fail_count);
  ctx->launches++;
  CK(ctx, cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------ introspection
extern "C" int zk_circuit_cols(int c) { return (c >= 0 && c < ZK_N_CIRCUITS) ? kCircuitCols[c] : -1; }
extern "C" int zk_table_cols(int t) { return (t >= 0 && t < ZK_N_TABLES) ? kTableCols[t] : -1; }
extern "C" int zk_n_constraints(int circuit) {
  int n = 0;
  circuit_info(circuit, &n);
  return n;
}
extern "C" int zk_constraint_info(int circuit, int idx, char* buf, int n) {
  int cnt = 0;
  const ConstraintInfo* info = circuit_info(circuit, &cnt);
  if (!info || idx < 0 || idx >= cnt) return -1;
  if (buf && n > 0) snprintf(buf, n, "%s: %s", info[idx].name, info[idx].doc);
  return info[idx].cls;
}
extern "C" uint64_t zk_launch_count(zk_ctx* ctx) { return ctx->launches; }
