/*
 * zkcheck.h — C-ABI of libzkcheck.so, the B200 constraint checker behind the
 * zkevm-specs Python API.
 *
 * The reference (privacy-scaling-explorations/zkevm-specs @ 6058c68) has no FFI;
 * its only seam is Python function signatures.  Each entry point below replaces
 * the INSIDE of one of those functions' per-row loops (file:line are relative to
 * the reference tree):
 *
 *   zk_check(ZK_CIRCUIT_BYTECODE) <- check_bytecode_row loop   src/zkevm_specs/bytecode_circuit.py:37-100
 *                                                              (driver: tests/test_bytecode_circuit.py:26-47)
 *   zk_check(ZK_CIRCUIT_STATE)    <- check_state_row loop      src/zkevm_specs/state_circuit.py:492-613
 *                                                              (driver: tests/test_state_circuit.py:17-38)
 *   zk_check(ZK_CIRCUIT_COPY)     <- verify_copy_table         src/zkevm_specs/copy_circuit.py:92-130
 *   zk_check(ZK_CIRCUIT_EVM)      <- verify_steps/verify_step  src/zkevm_specs/evm_circuit/main.py:14-63
 *   zk_upload_table / lookups     <- Tables + lookup()         src/zkevm_specs/evm_circuit/table.py:578-884
 *   zk_set_challenge              <- the `r` / keccak_randomness arguments of the functions above
 *
 * Data model
 *   cell   : one BN254-Fr element, CANONICAL (value < p), 4 little-endian uint64 limbs (32 B).
 *   column : n_rows consecutive cells.
 *   matrix : column-major, uint64[n_cols][n_rows][4]; a warp reading one column for 32
 *            consecutive rows touches 1 KiB of contiguous HBM.
 * All pointers are caller-owned HOST memory unless the name says "_device".  Nothing is
 * retained after a call returns except the device copies owned by the context.
 *
 * Return codes: 0 = the call ran (results are in the output arrays); < 0 = infrastructure
 * error (bad shape, missing table, CUDA error) — zk_last_error() has the text.
 * A context is not thread-safe; use one context per host thread / per GPU, and ONE stream per
 * context: uploads, index builds and checks are ordered only by the stream they are issued on
 * (cached lookup indexes are built on the stream of the first check that needs them).  Callers that
 * use several streams must order them with events themselves.
 * Cells must be canonical (< p): the reference's FQ() reduces on construction, the Python mirror
 * does the same before it ships a matrix; a raw caller that uploads unreduced 256-bit values gets
 * undefined verdicts (field add/sub assume a + b < 2^255).  Challenges are validated.
 */
#ifndef ZKCHECK_H
#define ZKCHECK_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct zk_ctx zk_ctx;

/* ---- circuits (witness matrices) -------------------------------------------------- */
enum {
  ZK_CIRCUIT_BYTECODE = 0, /* 12 cells/row, rotation {0,+1}     bytecode_circuit.py:15-27 */
  ZK_CIRCUIT_STATE = 1,    /* 57 cells/row, rotation {-1,0,+1}  state_circuit.py:63-96    */
  ZK_CIRCUIT_COPY = 2,     /* 20 cells/row, rotation {0,+1,+2}  evm_circuit/table.py:472-491 */
  ZK_CIRCUIT_EVM = 3,      /* 13 cells/step, rotation {0,+1}    evm_circuit/step.py:16-44 */
  ZK_CIRCUIT_EXP = 4,      /* 21 cells/row, rotation {0,+1}     evm_circuit/table.py:519-535 */
  ZK_CIRCUIT_TX = 5,       /* 14 cells/row, no rotation: one row per tx_index = SignVerifyChip cells
                              (address, pub_key_x lo/hi, pub_key_y lo/hi, Word(pub_key_hash) lo/hi, msg_hash
                              lo/hi, Word(msg_hash_bytes) lo/hi — a 32-byte field travels as the Word of its
                              bytes) + the tx-table cells they are copy-constrained to (CallerAddress value,
                              TxSignHash lo/hi)
                              tx_circuit.py:160-243, 253-289; row flags bit 0 = the CallerAddress
                              cell is a Word, bit 1 = the (third-party) ECDSA check failed;
                              lookups: ZK_TABLE_KECCAK rows (is_enabled, input_rlc, input_len, out lo, hi) */
  ZK_CIRCUIT_SIG = 6,      /* 21 cells/row, no rotation: sig_circuit.Row (sig_circuit.py:7-49): sig_v,
                              recovered_addr, pub_key_x lo/hi, pub_key_y lo/hi, Word(pub_key_hash) lo/hi,
                              msg_hash lo/hi, Word(msg_hash_bytes) lo/hi, is_valid, sig_r lo/hi, sig_s
                              lo/hi, the ECDSA chip's r lo/hi and s lo/hi; row flags bit 1 = the
                              (third-party) ecdsa_chip.verify() returned True; same keccak table */
  ZK_CIRCUIT_PI = 7,       /* 28 cells/row, rotation {0,+1}: pi_circuit.Row (pi_circuit.py:105-133), Words as (lo, hi), the
                              tx-table and withdrawal-table rows a Row carries flattened behind it: q_bytes_last,
                              q_tx_table, q_tx_calldata, q_tx_calldata_start, q_rpi_keccak_lookup, q_rpi_value_start,
                              tx_id_inv, tx_value_lo_inv, tx_id_diff_inv, calldata_gas_cost, is_final,
                              q_withdrawal_table, rpi_bytes, rpi_bytes_keccakrlc, rpi_value_lc, rpi_digest_word lo/hi,
                              q_rpi_byte_enable, tx (tx_id, tag, index, value lo/hi), withdrawal (id, validator_id,
                              address lo/hi, amount); lookups: ZK_TABLE_KECCAK, ZK_TABLE_CALLDATA_GAS; parameters:
                              ZK_CHALLENGE_PI_KECCAK, ZK_CHALLENGE_PI_BYTE_BASE, ZK_PARAM_PI_CIRCUIT_LEN */
  ZK_CIRCUIT_WITHDRAWAL = 8, /* 8 cells/row, rotation {-1,0,+1} without wrap: withdrawal_circuit.Row (withdrawal_circuit.py:20-44):
                              withdrawal_id, validator_id, address, amount, hash lo/hi, root lo/hi.  Global row 0 has no
                              predecessor (root_prev = Word(0)); global row ZK_PARAM_WITHDRAWAL_MAX - 1 has no successor and
                              owns the block-table lookup; rows at or past MAX are not part of the circuit.  lookups:
                              ZK_TABLE_KECCAK (5 columns), ZK_TABLE_MPT (12 columns), ZK_TABLE_BLOCK (field_tag, value lo,
                              hi); parameters: ZK_CHALLENGE_KECCAK (the RLC of the RLP bytes), ZK_PARAM_WITHDRAWAL_MAX */
  ZK_N_CIRCUITS = 9
};

/* ---- lookup tables ---------------------------------------------------------------- */
enum {
  ZK_TABLE_FIXED = 0,    /* 4 cells  FixedTableRow     table.py:405-409 */
  ZK_TABLE_BYTECODE = 1, /* 6 cells  BytecodeTableRow  table.py:438-443 (hash lo,hi,tag,index,is_code,value) */
  ZK_TABLE_RW = 2,       /* 14 cells RWTableRow        table.py:447-457 */
  ZK_TABLE_TX = 3,       /* 5 cells  TxTableRow        table.py:421-426 (tx_id,tag,index,value lo,hi) */
  ZK_TABLE_BLOCK = 4,    /* 4 cells  BlockTableRow     table.py:413-417 */
  ZK_TABLE_COPY = 5,     /* 14 cells CopyTableRow      table.py:495-507 */
  ZK_TABLE_KECCAK = 6,   /* 5 cells  KeccakTableRow    table.py:511-515 (state_tag,input_rlc,input_len,out lo,hi) */
  ZK_TABLE_MPT = 7,      /* 12 cells MPTTableRow       table.py:460-468 */
  ZK_TABLE_PUSH = 8,     /* 2 cells  push table        bytecode_circuit.py:174-178 (byte, push_size) */
  ZK_TABLE_WITHDRAWAL = 9, /* 4 cells WithdrawalTableRow table.py:429-435 (id, validator_id, address, amount) */
  ZK_TABLE_CALLDATA_GAS = 10, /* 3 cells TxCallDataGasCostAccRow pi_circuit.py:66-70 (tx_id, is_final, gas_cost_acc) */
  ZK_TABLE_EXP = 11,     /* 11 cells ExpTableRow     table.py:539-548 (is_step, identifier, is_last, base limbs 0..3, exponent lo,hi,
                            exponentiation lo,hi) */
  ZK_TABLE_STEP_AUX = 12, /* 3 cells  StepState.aux_data  step.py (step row, aux lo, hi): the per-step auxiliary word CREATE / CREATE2
                            read as the init code's hash (create.py:107); rows only for the steps that carry one */
  ZK_N_TABLES = 13
};

/* ---- challenges ------------------------------------------------------------------- */
enum {
  ZK_CHALLENGE_KECCAK = 0, /* keccak_randomness / `r` of bytecode & copy circuits */
  ZK_CHALLENGE_LOOKUP = 1, /* RLC base used to compress table rows into hash keys;
                              any value gives the same pass/fail (matches are confirmed
                              exactly), it only affects bucket placement */
  ZK_CHALLENGE_PI_KECCAK = 2,    /* pi_circuit.keccak_rand (a module global of the reference, pi_circuit.py:836) */
  ZK_CHALLENGE_PI_BYTE_BASE = 3, /* pi_circuit.byte_pow_base (pi_circuit.py:834) */
  ZK_PARAM_PI_CIRCUIT_LEN = 4,   /* Witness.circuit_len (pi_circuit.py:333), a circuit parameter held like a challenge */
  ZK_PARAM_WITHDRAWAL_MAX = 5,   /* MAX_WITHDRAWALS of withdrawal_circuit.verify_circuit (:130), below 2^32: tells a row
                                    shard (row_base) which global row is the last one */
  ZK_N_CHALLENGES = 6
};

/* ---- zk_check flags ---------------------------------------------------------------- */
enum {
  ZK_FLAG_WRAP = 1,             /* rotations wrap modulo n_rows (whole circuit resident) */
  ZK_FLAG_EVM_FIRST_STEP = 2,   /* verify_steps(begin_with_first_step=True)  main.py:30 */
  ZK_FLAG_EVM_LAST_STEP = 4     /* verify_steps(end_with_last_step=True): the caller has
                                   appended the dummy EndBlock step           main.py:21-22 */
};

/* ---- error classes a constraint id maps to (SURVEY.md Appendix B) ------------------- */
enum {
  ZK_ERR_ASSERT = 0,           /* AssertionError — caught by verify_steps (main.py:45)   */
  ZK_ERR_LOOKUP_UNSAT = 1,     /* LookupUnsatFailure      table.py:879                  */
  ZK_ERR_LOOKUP_AMBIGUOUS = 2, /* LookupAmbiguousFailure  table.py:881                  */
  ZK_ERR_RANGE_RAISE = 3,      /* ConstraintUnsatFailure raised (instruction.py:529-534) */
  ZK_ERR_VALUE = 4,            /* ValueError / OverflowError from Python runtime          */
  ZK_ERR_NOT_IMPLEMENTED = 5   /* NotImplementedError (main.py:63) or a state this build
                                  has no gate program for                                */
};

#define ZK_PASS 0xFFFFFFFFu /* first_fail value meaning "constraint held on every row" */

/* lifecycle */
int zk_ctx_create(int device_ordinal, zk_ctx** out);
void zk_ctx_destroy(zk_ctx* ctx);
const char* zk_last_error(zk_ctx* ctx); /* ctx may be NULL: last create error */

/* canonical Fr challenge, 4 LE limbs */
int zk_set_challenge(zk_ctx* ctx, int which, const uint64_t r[4]);

/* Witness matrix of one circuit: host uint64[n_cols][n_rows][4]; n_cols must equal the
 * circuit's cell count (zk_circuit_cols).  Copies host->device on `stream` (a cudaStream_t
 * passed as void*, NULL = default stream). */
int zk_upload_columns(zk_ctx* ctx, int circuit_id, uint64_t n_rows, uint32_t n_cols,
                      const uint64_t* colmajor, void* stream);
/* Same, but the matrix already lives in device memory (e.g. a torch tensor); the context
 * borrows the pointer until the next upload/bind for this circuit. */
int zk_bind_columns_device(zk_ctx* ctx, int circuit_id, uint64_t n_rows, uint32_t n_cols,
                           const uint64_t* colmajor_device);

/* Optional per-row type flags that the Python objects carry outside the cells
 * (WordOrValue.is_word, arithmetic.py:171-189): one byte per row, bit k = "word k of the
 * row is a Word".  NULL / never called = all zero. Host pointer. */
int zk_upload_row_flags(zk_ctx* ctx, int circuit_id, uint64_t n_rows, const uint8_t* flags,
                        void* stream);

/* Lookup table: host uint64[n_cols][n_rows][4].  Any index built on the previous contents
 * is dropped; it is rebuilt on the device by the next zk_check that needs it. */
int zk_upload_table(zk_ctx* ctx, int table_id, uint64_t n_rows, uint32_t n_cols,
                    const uint64_t* colmajor, void* stream);
int zk_bind_table_device(zk_ctx* ctx, int table_id, uint64_t n_rows, uint32_t n_cols,
                         const uint64_t* colmajor_device);
int zk_upload_table_flags(zk_ctx* ctx, int table_id, uint64_t n_rows, const uint8_t* flags,
                          void* stream);

/* Packed columns — the compact host format of the same matrices.  The reference's cells are
 * Python ints, most of them bytes, flags, tags and counters (table.py:405-535 row types); a
 * packer that knows (or measures) each column's range hands column c over as n_rows
 * little-endian unsigned integers of col_widths[c] bytes, col_widths[c] in {1,2,4,8,16,32};
 * 0 = constant column, stored once as one 32-byte cell.  `packed` is ONE host buffer of
 * total_bytes; column c starts at byte col_offsets[c] (a multiple of 32).  The buffer is
 * copied host->device as it is and the kernels read the narrow columns in place (no widening
 * pass), so both the PCIe bytes and the HBM bytes of a check shrink with the data.
 * A 32-byte column holds canonical cells exactly as in zk_upload_columns.  Results are
 * identical to the canonical upload of the same values (tests/test_gpu_packed.py). */
int zk_upload_columns_packed(zk_ctx* ctx, int circuit_id, uint64_t n_rows, uint32_t n_cols,
                             const void* packed, uint64_t total_bytes,
                             const uint64_t* col_offsets, const uint8_t* col_widths, void* stream);
int zk_upload_table_packed(zk_ctx* ctx, int table_id, uint64_t n_rows, uint32_t n_cols,
                           const void* packed, uint64_t total_bytes,
                           const uint64_t* col_offsets, const uint8_t* col_widths, void* stream);

/* The bytecode table from the bytecode itself.  Replaces Bytecode.table_assignments
 * (src/zkevm_specs/evm_circuit/typing.py:390-427) + the column packer for ZK_TABLE_BYTECODE: the
 * reference unrolls every contract into one Header row (hash, Header, 0, 0, len) and len Byte rows
 * (hash, Byte, i, is_code[i], code[i]) on the host; here the host ships only the code bytes, one
 * is_code BIT per byte and one hash per contract, and the six columns are written on the device
 * (k_bytecode_table_expand), in contract order, as a packed table [16,16,1,4,1,4].  ~1.1 bytes
 * cross PCIe per table row instead of 192 (canonical) or 10-42 (packed).
 *   code          : concatenated code bytes of all contracts
 *   is_code_bits  : bit j (LSB first within a byte) = is_code of concatenated byte j
 *                   (Bytecode.is_code, typing.py:309-386: false for PUSH data)
 *   code_offsets  : [n_contracts + 1], contract k = bytes [code_offsets[k], code_offsets[k+1])
 *   hashes        : [n_contracts][4] = code hash as (lo limb0, lo limb1, hi limb0, hi limb1)
 * The result is an ordinary resident table (same lookups, same index building / verification). */
int zk_upload_bytecode_table_from_code(zk_ctx* ctx, uint64_t n_contracts, const uint8_t* code,
                                       const uint8_t* is_code_bits, const uint64_t* code_offsets,
                                       const uint64_t* hashes, void* stream);

/* Keccak-256 on the device (original 0x01 padding).  The reference hashes on the host through third-party
 * packages (src/zkevm_specs/util/hash.py:7-10); its witness generators need one digest per contract and per
 * copy event.  Message k = data[offsets[k] .. offsets[k+1]).
 *   zk_keccak256_batch     : digests[k][0..3] = the 32 digest bytes of message k as four little-endian uint64 lanes
 *   zk_assign_keccak_table : KeccakCircuit.add / assign_keccak_table (evm_circuit/typing.py:854-865,
 *                            bytecode_circuit.py:182-186) for every message: the resident ZK_TABLE_KECCAK becomes
 *                            n rows (2, RLC of the bytes under ZK_CHALLENGE_KECCAK, length, hash lo, hash hi),
 *                            hashed and folded on the device; nothing but the message bytes crosses PCIe */
int zk_keccak256_batch(zk_ctx* ctx, uint64_t n, const uint8_t* data, const uint64_t* offsets, uint64_t* digests, void* stream);
int zk_assign_keccak_table(zk_ctx* ctx, uint64_t n, const uint8_t* data, const uint64_t* offsets, void* stream);

/* ---- witness assignment on the device (SURVEY.md 8(f)-3; csrc/assign.cu) ------------------------------------
 * The reference builds circuit rows with Python object loops; these calls expand the compact data those
 * loops start from into the resident witness matrix of a circuit, stored as narrow columns, ready for zk_check.
 *
 * zk_assign_bytecode_circuit = assign_bytecode_circuit (bytecode_circuit.py:104-167): 2^k rows from the raw code of
 *   n_contracts contracts (arguments as zk_upload_bytecode_table_from_code: code bytes, one is_code bit per byte as
 *   Bytecode.table_assignments computes it, code_offsets[n + 1], hashes[n][4] = hash lo (2 limbs), hi (2 limbs)):
 *   Header + Byte rows of every contract in order, truncated at 2^k rows, then (EMPTY_HASH, Header) padding;
 *   value_rlc under ZK_CHALLENGE_KECCAK.
 * zk_assign_state_circuit = op2row of every operation (state_circuit.py:827-857): `packed_ops` holds the 15 cells
 *   an operation brings (rw_counter, is_write, tag, id, address, field_tag, storage_key lo, hi, value lo, hi,
 *   initial_value lo, hi, root lo, hi, lexicographic_ordering_selector) in the packed column format
 *   (zk_upload_columns_packed); the ten 16-bit address limbs and the 32 storage-key bytes of the 57-cell row are
 *   derived on the device.  An address beyond 160 bits is an error (the reference raises OverflowError).
 *   row_flags as zk_upload_row_flags (may be NULL).
 * zk_assign_copy_circuit = CopyCircuit.copy per event (evm_circuit/typing.py:1010-1147): events[n][16] =
 *   { src_tag | src id is a Word << 8, dst_tag | dst id is a Word << 8, src_addr, src_addr_end, dst_addr, copy_length,
 *   log_id, rw_counter before the event, src_id lo (2 limbs), hi (2 limbs), dst_id lo (2 limbs), hi (2 limbs) };
 *   `data` = the copied byte values of all events back to back (copy_length bytes each, 0 where the source address is
 *   at or beyond src_addr_end), is_code_bits = one bit per data byte (events that touch bytecode; may be NULL).
 *   Two rows per byte (read row, write row) incl. rlc_acc under ZK_CHALLENGE_KECCAK, rw_counter / rwc_inc_left and
 *   the id type flags.
 * zk_download_columns widens the resident matrix of a circuit back to canonical cells
 *   (colmajor_out: uint64[n_cols][zk_resident_rows][4]; flags_out: uint8[rows] or NULL) — inspection and tests. */
int zk_assign_bytecode_circuit(zk_ctx* ctx, uint32_t k, uint64_t n_contracts, const uint8_t* code, const uint8_t* is_code_bits,
                               const uint64_t* code_offsets, const uint64_t* hashes, void* stream);
int zk_assign_state_circuit(zk_ctx* ctx, uint64_t n_rows, const void* packed_ops, uint64_t total_bytes,
                            const uint64_t* col_offsets, const uint8_t* col_widths, const uint8_t* row_flags, void* stream);
int zk_assign_copy_circuit(zk_ctx* ctx, uint64_t n_events, const uint64_t* events, const uint8_t* data,
                           const uint8_t* is_code_bits, void* stream);
/* zk_assign_withdrawal_circuit = withdrawals2witness (the reference's tests/test_withdrawal_circuit.py:27-96) on the
 *   device: records[n][5][4] = withdrawal_id, validator_id, address, amount as canonical cells and the MPT root as a
 *   256-bit word (4 little-endian limbs, stored as root lo / hi).  The resident
 *   ZK_CIRCUIT_WITHDRAWAL matrix becomes max_withdrawals rows (n <= max_withdrawals): row k < n = the record with
 *   hash = Word(keccak256(rlp([id, validator_id, address, amount]))), rows n.. = Row(0, 0, 0, 0, Word(0), last root)
 *   (last root = root of record n - 1, 0 if n == 0).  The resident ZK_TABLE_KECCAK becomes the all-zero row followed by
 *   one row (1, RLC of the RLP bytes under ZK_CHALLENGE_KECCAK, length, hash lo, hash hi) per record.  The MPT and
 *   block tables are the caller's (uploads). */
int zk_assign_withdrawal_circuit(zk_ctx* ctx, uint64_t n, const uint64_t* records, uint64_t max_withdrawals, void* stream);
int64_t zk_resident_rows(zk_ctx* ctx, int circuit_id);
int zk_download_columns(zk_ctx* ctx, int circuit_id, uint64_t* colmajor_out, uint8_t* flags_out, void* stream);

/* Check rows [row_begin, row_end) of the resident matrix (local indices).  Without
 * ZK_FLAG_WRAP the caller guarantees halo rows exist for the circuit's rotations.
 * Reported rows are row_base + local index.
 *   first_fail[n]  : per constraint id, the smallest failing row, ZK_PASS if none
 *   fail_count[n]  : optional (may be NULL) number of failing rows per constraint
 * n = zk_n_constraints(circuit_id).  The call enqueues on `stream`, then copies the two
 * arrays back and synchronises the stream. */
int zk_check(zk_ctx* ctx, int circuit_id, uint64_t row_begin, uint64_t row_end,
             uint64_t row_base, uint32_t flags, uint32_t* first_fail, uint64_t* fail_count,
             void* stream);

/* Asynchronous form used for device-side timing and multi-GPU: enqueues the index builds
 * and the check kernels on `stream` and leaves the result in device memory owned by the
 * context.  (ZK_CIRCUIT_EVM: the call waits on the host until the step-classification kernel has
 * finished — it reads the per-state step counts back to launch only the gate-program kernels that
 * have work — and returns with those kernels still running.)  zk_result_device returns that buffer (uint32 first_fail[n] followed, 8-byte
 * aligned, by uint64 fail_count[n]) so a collective can reduce it in place; zk_fetch_result
 * copies it to the host and synchronises. */
int zk_check_async(zk_ctx* ctx, int circuit_id, uint64_t row_begin, uint64_t row_end,
                   uint64_t row_base, uint32_t flags, void* stream);
int zk_result_device(zk_ctx* ctx, int circuit_id, uint32_t** first_fail_device,
                     uint64_t** fail_count_device);
int zk_fetch_result(zk_ctx* ctx, int circuit_id, uint32_t* first_fail, uint64_t* fail_count,
                    void* stream);

/* Multi-GPU: element-wise MIN of first_fail and SUM of fail_count across the ranks of an NCCL
 * communicator (ncclComm_t passed as void*), on `stream`, in place in the context's device result
 * buffer (read it with zk_fetch_result).  ONE collective — the ranks' result vectors (a few KB) are
 * all-gathered and folded by a one-block kernel; rows are sharded, tables replicated, so this is the
 * only exchange (SURVEY.md §8e). */
int zk_allreduce_results(zk_ctx* ctx, int circuit_id, void* nccl_comm, void* stream);
/* Communicator plumbing for callers whose host language has no NCCL binding: rank 0 draws the
 * 128-byte unique id, ships it to the other ranks by whatever means it has (MPI, a socket, gloo),
 * every rank then joins.  NCCL itself is bound at run time (dlopen of libnccl.so.2). */
int zk_nccl_unique_id(zk_ctx* ctx, uint8_t id[128]);
int zk_nccl_comm_init(zk_ctx* ctx, int world_size, int rank, const uint8_t id[128], void** comm_out);
int zk_nccl_comm_destroy(zk_ctx* ctx, void* comm);

/* introspection */
int zk_circuit_cols(int circuit_id);
int zk_table_cols(int table_id);
int zk_n_constraints(int circuit_id);
/* name into buf (NUL-terminated, truncated to n); returns the ZK_ERR_* class, <0 if bad id */
int zk_constraint_info(int circuit_id, int idx, char* buf, int n);
/* number of kernels this context has launched since creation (bench.py: gpu_launches) */
uint64_t zk_launch_count(zk_ctx* ctx);
/* Device-side timing of the two phases of a check (lookup-index builds, then the circuit
 * kernel), measured with CUDA events recorded on the SAME stream the kernels are launched on.
 * zk_enable_timing(ctx, 1) makes every zk_check_async record events; zk_last_timing returns
 * the durations of the most recent check after synchronising its events (milliseconds). */
int zk_enable_timing(zk_ctx* ctx, int on);
int zk_last_timing(zk_ctx* ctx, float* index_build_ms, float* check_kernel_ms);
/* drop the cached lookup indexes of the witness tables so the next zk_check rebuilds them (used
 * by bench to time the whole path); the fixed table is a circuit constant (table.py:37-103,
 * uploaded once), its index lives until the table is uploaded again */
int zk_invalidate_indexes(zk_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* ZKCHECK_H */
