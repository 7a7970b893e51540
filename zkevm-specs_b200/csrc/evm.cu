// evm.cu — EVM-circuit step checker.
//
// Replaces the loop body of verify_steps / verify_step
// (src/zkevm_specs/evm_circuit/main.py:14-63): state-transition legality
// (instruction.py:189-204), one gate program per execution state, and the shared epilogue
// step_state_transition_in_same_context (instruction.py:365-394, 206-264).
// Hot gate programs (a kernel each): ADD/SUB (execution/add_sub.py:5-24), MUL/DIV/MOD
// (mul_div_mod.py:6-71 with mul_add_words instruction.py:599-632 and compare_word :453-463), PUSH
// (push.py:6-33), POP (pop.py:4-14).  Rare gate programs (k_evm_misc, one thread per step, out-of-line
// lookups): SHA3, CALLDATACOPY, MEMORY, STOP with restore-to-caller-context, MSIZE, GAS, ISZERO, CMP, JUMP,
// JUMPI, CALLER, CALLVALUE, CALLDATASIZE, ADDRESS, RETURNDATASIZE, CODESIZE, BITWISE, NOT, BYTE, SCMP,
// SIGNEXTEND, BlockCtx, ORIGIN, GASPRICE, SHL_SHR (their execution/*.py files, cited at each program).
// Every lookup() of the reference (table.py:864-884, a linear scan over a Python set) is either a
// positional lookup on a verified-regular table or a probe of a device hash index (lookup.cuh).
//
// Step = 13 cells in the order of StepState (evm_circuit/step.py:16-44), code_hash as
// (lo, hi); rotation {0,+1}.  Algorithmic bytes per step: 13 x 32 B = 416 B, plus the
// table rows it touches, counted once per table row (rw 448 B, bytecode 192 B).
// A step stops at its first failing constraint (the reference raises there), so at most one
// constraint id is recorded per step.
#include "circuit.cuh"
#include "keccak.cuh"
#include "words.cuh"
#include "../../include/zk_constraints.h"
#include "../../include/zk_evm_spec.h"
#include "../../include/zkcheck.h"

namespace zk {

enum { S_STATE, S_RWC, S_CALL_ID, S_IS_ROOT, S_IS_CREATE, S_HASH_LO, S_HASH_HI, S_PC, S_SP, S_GAS,
       S_MEM, S_REV, S_LOG };
enum { B_HASH_LO, B_HASH_HI, B_TAG, B_INDEX, B_ISCODE, B_VALUE };
enum { R_RWC, R_RW, R_TAG, R_ID, R_ADDR, R_FIELD, R_KEY_LO, R_KEY_HI, R_VAL_LO, R_VAL_HI };

// execution states with a gate program in this build (others: EV_UNSUPPORTED_STATE)
#define ZK_ES_BUILT_LIST(X)                                                                                            \
  X(ZK_ES_ADD) X(ZK_ES_MUL) X(ZK_ES_PUSH) X(ZK_ES_POP) X(ZK_ES_SHA3) X(ZK_ES_CALLDATACOPY) X(ZK_ES_STOP) X(ZK_ES_MEMORY)  \
  X(ZK_ES_MSIZE) X(ZK_ES_GAS) X(ZK_ES_ISZERO) X(ZK_ES_CMP) X(ZK_ES_JUMP) X(ZK_ES_JUMPI) X(ZK_ES_CALLER) X(ZK_ES_CALLVALUE) \
  X(ZK_ES_CALLDATASIZE) X(ZK_ES_ADDRESS) X(ZK_ES_RETURNDATASIZE) X(ZK_ES_CODESIZE) X(ZK_ES_BITWISE) X(ZK_ES_NOT)         \
  X(ZK_ES_BYTE) X(ZK_ES_SCMP) X(ZK_ES_SIGNEXTEND) X(ZK_ES_BlockCtx) X(ZK_ES_ORIGIN) X(ZK_ES_GASPRICE) X(ZK_ES_SHL_SHR)      \
  X(ZK_ES_BeginTx) X(ZK_ES_EndTx) X(ZK_ES_EndBlock) X(ZK_ES_ErrorStack) X(ZK_ES_ErrorInvalidOpcode)                    \
  X(ZK_ES_ErrorOutOfGasConstant) X(ZK_ES_ErrorInvalidJump) X(ZK_ES_SELFBALANCE) X(ZK_ES_ErrorOutOfGasSHA3)                  \
  X(ZK_ES_ErrorOutOfGasStaticMemoryExpansion) X(ZK_ES_ErrorOutOfGasDynamicMemoryExpansion) X(ZK_ES_ErrorOutOfGasLOG)       \
  X(ZK_ES_ErrorOutOfGasEXP) X(ZK_ES_ErrorReturnDataOutOfBound) X(ZK_ES_BALANCE) X(ZK_ES_EXTCODEHASH) X(ZK_ES_EXTCODESIZE)          \
  X(ZK_ES_ErrorOutOfGasAccountAccess) X(ZK_ES_CODECOPY) X(ZK_ES_RETURNDATACOPY) X(ZK_ES_EXTCODECOPY) X(ZK_ES_ErrorOutOfGasMemoryCopy) \
  X(ZK_ES_ADDMOD) X(ZK_ES_MULMOD) X(ZK_ES_SDIV_SMOD) X(ZK_ES_SAR) X(ZK_ES_SLOAD) X(ZK_ES_SSTORE) X(ZK_ES_CALLDATALOAD) \
  X(ZK_ES_LOG) X(ZK_ES_ErrorWriteProtection) X(ZK_ES_BLOCKHASH) X(ZK_ES_EXP) \
  X(ZK_ES_ErrorMaxCodeSizeExceeded) X(ZK_ES_ErrorOutOfGasCodeStore) X(ZK_ES_ErrorInvalidCreationCode) X(ZK_ES_RETURN) X(ZK_ES_ErrorOutOfGasCall) X(ZK_ES_CALL_OP) \
  X(ZK_ES_CREATE) X(ZK_ES_CREATE2) X(ZK_ES_ErrorOutOfGasSloadSstore) X(ZK_ES_ErrorOutOfGasCREATE) X(ZK_ES_ErrorOutOfGasPrecompile) \
  X(ZK_ES_ErrorGasUintOverflow)
struct EsBuiltTable {
  signed char v[ZK_ES_COUNT];
};
__host__ __device__ constexpr EsBuiltTable make_es_built() {
  EsBuiltTable t{};
#define ZK_X(id) t.v[id] = 1;
  ZK_ES_BUILT_LIST(ZK_X)
#undef ZK_X
  return t;
}
#ifdef __CUDACC__
__constant__ EsBuiltTable c_es_built = make_es_built();
__constant__ signed char c_es_halts[ZK_ES_COUNT] = ZK_ES_HALTS_INIT;
__constant__ signed char c_es_impl[ZK_ES_COUNT] = ZK_ES_IMPLEMENTED_INIT;
__constant__ short c_opcode_gas[256] = ZK_OPCODE_GAS_INIT;
#endif
static const EsBuiltTable h_es_built = make_es_built();
static const signed char h_es_halts[ZK_ES_COUNT] = ZK_ES_HALTS_INIT;  // host copies: tests/emu only
static const signed char h_es_impl[ZK_ES_COUNT] = ZK_ES_IMPLEMENTED_INIT;
static const short h_opcode_gas[256] = ZK_OPCODE_GAS_INIT;
#ifdef __CUDA_ARCH__
#define ES_BUILT(i) c_es_built.v[i]
#define ES_HALTS(i) c_es_halts[i]
#define ES_IMPL(i) c_es_impl[i]
#define OPCODE_GAS(i) c_opcode_gas[i]
#else
#define ES_BUILT(i) h_es_built.v[i]
#define ES_HALTS(i) h_es_halts[i]
#define ES_IMPL(i) h_es_impl[i]
#define OPCODE_GAS(i) h_opcode_gas[i]
#endif

// constants in Montgomery form: montmul(x, C*2^256) == x*C mod p
#define ZK_MONT_INV8 Fr{{0x0ull, 0x0ull, 0x0ull, 0x2000000000000000ull}}
#define ZK_MONT_INV4 Fr{{0xbc1e0a6c0fffffffull, 0xd7cc17b786468f6eull, 0x47afba497e7ea7a2ull, 0x0f9bb18d1ece5fd6ull}}

struct EvmTables {
  IndexDev bytecode;  // key (hash_lo, hash_hi, tag, index, is_code)
  IndexDev rw;        // key (rw_counter, rw, tag, id, address)
  IndexDev fixed;     // key (tag, v0, v1, v2)
  IndexDev copy;      // copy table, key = every queried cell of copy_lookup (table.py:760-787): cells 1..10, 12
  IndexDev keccak;    // keccak table, key (state_tag, input_rlc, input_len)
  IndexDev tx;        // tx table (tx_id, tag, index | value lo, hi), key = the first three cells (table.py:697-705)
  IndexDev block;     // block table (tag, block number | value lo, hi), key = the first two cells (table.py:691-695)
  IndexDev exp;       // exp table (is_step, identifier, is_last, base limbs 0..3, exponent lo / hi | exponentiation lo / hi), key = the
                      // first nine cells (table.py:797-814)
  IndexDev aux;       // step-aux side table (step row | aux_data lo, hi): StepState.aux_data of CREATE / CREATE2 (create.py:107), key =
                      // the step's row
  IndexDev bytecode4; // bytecode table keyed on (hash lo, hi, tag, index): bytecode_lookup_pair does not name is_code; only built
                      // when an ErrorInvalidJump step exists and the bytecode table is not positional
  IndexDev rw_rwc;    // rw table keyed on rw_counter alone: lookups that name other column subsets (evm_tx.cuh);
                      // only built when a BeginTx / EndTx / EndBlock step exists and the rw table is not positional
  TableDev wd;        // withdrawal table (id, validator_id, address, amount), table.py:429-435
  const struct BlockStats* stats;  // table-derived constants of EndBlock (k_evm_block_stats)
  // ResponsibleOpcode rows of the fixed table (tag 13, aux 0) with state, opcode < 256 as a
  // 64 Kbit bitmap: bit (state << 8 | opcode).  Built from the uploaded fixed table
  // (k_fixed_resp_bitmap) and staged into shared memory by every EVM kernel.
  const u32* resp_bitmap;
};
#define ZK_RESP_BITMAP_WORDS 2048

// one thread per fixed-table row
ZK_HD void resp_bitmap_row(const TableDev& fixed, u32* bitmap, u64 row) {
  const Fr tag = table_cell(fixed, 0, row), st = table_cell(fixed, 1, row);
  const Fr op = table_cell(fixed, 2, row), aux = table_cell(fixed, 3, row);
  if (fr_eq_u64(tag, ZK_FIXED_ResponsibleOpcode) && fr_is_zero(aux) && fr_fits64(st) && st.l[0] < 256 &&
      fr_fits64(op) && op.l[0] < 256) {
    const u32 bit = (u32)(st.l[0] << 8 | op.l[0]);
#ifdef __CUDA_ARCH__
    atomicOr(&bitmap[bit >> 5], 1u << (bit & 31));
#else
    bitmap[bit >> 5] |= 1u << (bit & 31);
#endif
  }
}
#ifdef __CUDACC__
__global__ void __launch_bounds__(256) k_fixed_resp_bitmap(TableDev fixed, u32* bitmap) {
  const u64 row = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (row < fixed.n_rows) resp_bitmap_row(fixed, bitmap, row);
}
#endif

// per-thread view of one step
struct StepCtx {
  const WitnessDev& w;
  const EvmTables& t;
  const ResultDev& res;
  u64 i, j, row;
  bool record;      // warp-cooperative gadgets evaluate in every lane but only one lane records
  const u32* resp;  // ResponsibleOpcode bitmap (shared memory on the device)
  unsigned mask;    // lanes that run this gate program together (warp-synchronous lookups)
  const Fr* stack_pre;  // [2]: rw * r + Target.Stack * r^2 for rw = Read, Write (constant key terms)
  const u64* rw_base;  // limb 0 of rw_counter of rw-table row 0, hoisted (positional rw table), or nullptr
  int pos_mode;  // -1: read the tables' positional flags at run time; 1: the kernel was specialised for
                 // positional rw + bytecode tables (the caller checked both flags), hash paths compiled out
  int narrow = 0;  // 1: the kernel instance runs only when the host found (api.cu:evm_narrow) every step column but the code
                   // hash, and the rw table's five key columns, narrow (<= 8 bytes per row) and the bytecode table in the
                   // layout k_bytecode_table_expand writes: those cells load as one limb with literal zero upper limbs
  ZK_HD Fr cur(u32 c) const {
    if (narrow == 1 && c != S_HASH_LO && c != S_HASH_HI) return ld_col_narrow(w.base + w.off[c], w.width[c], i);
    return wcell(w, c, i);
  }
  ZK_HD Fr nxt(u32 c) const {
    if (narrow == 1 && c != S_HASH_LO && c != S_HASH_HI) return ld_col_narrow(w.base + w.off[c], w.width[c], j);
    return wcell(w, c, j);
  }
};

ZK_HD void step_fail(const StepCtx& s, int id) {
  if (s.record) fail(s.res, id, s.row);
}
#define EV_CHECK(id, cond) \
  do {                     \
    if (!(cond)) {         \
      step_fail(s, (id));  \
      return;              \
    }                      \
  } while (0)
#define EV_CHECK_RET(id, cond, ret) \
  do {                              \
    if (!(cond)) {                  \
      step_fail(s, (id));           \
      return ret;                   \
    }                               \
  } while (0)

// lookup outcome -> failure id (unsat, or the next id = ambiguous); true iff exactly one row
ZK_HD bool need1(const StepCtx& s, bool live, int n, int id_unsat) {
  if (!live) return false;
  if (n == 1) return true;
  step_fail(s, n == 0 ? id_unsat : id_unsat + 1);
  return false;
}

// Lookups are warp-synchronous (lookup.cuh): every lane of s.mask calls them in the same order;
// `live` is false for lanes with nothing to look up (no step, or the step already failed).
ZK_HD int bytecode_lookup(const StepCtx& s, bool live, const Fr& hlo, const Fr& hhi, u64 tag, const Fr& index,
                          u64 is_code, Fr* value) {
  Fr key[5] = {hlo, hhi, fr_u64(tag), index, fr_u64(is_code)};
  u32 r;
  if (s.pos_mode == 1) {  // kernel specialised for positional tables: no hash code at all
    const IndexDev& ix = s.t.bytecode;
    u32 head = 0, len = 0;
    const int n_head = heads_probe(ix, hlo, hhi, &head, &len, s.mask, live);
    Fr got;
    const int n = s.narrow == 1 ? pos_lookup_run<true>(ix, key, n_head, head, len, &r, live, B_VALUE, &got)
                                : pos_lookup_run<false>(ix, key, n_head, head, len, &r, live, B_VALUE, &got);
    if (live && n == 1) *value = got;
    return n;
  }
  const int n = lookup_sync<5>(s.t.bytecode, key, &r, s.mask, live);
  if (live && n == 1) *value = table_cell(s.t.bytecode.tab, B_VALUE, r);
  return n;
}
// same lookup with the step-constant part of the key hash (hash_lo + hash_hi * r) hoisted: a PUSH
// step probes the bytecode table up to 34 times with the same code hash
ZK_HD Fr bytecode_hash0(const StepCtx& s, const Fr& hlo, const Fr& hhi) {
  return fr_add(hlo, rlc_term(s.t.bytecode, hhi, 1));
}
// `n_head/head`: result of the heads-index probe for this code hash (positional path), done once
// per step by the caller
ZK_HD int bytecode_lookup_h(const StepCtx& s, bool live, const Fr& h0, int n_head, u32 head, u32 run_len, const Fr& hlo,
                            const Fr& hhi, u64 tag, const Fr& index, u64 is_code, Fr* value) {
  Fr key[5] = {hlo, hhi, fr_u64(tag), index, fr_u64(is_code)};
  const IndexDev& ix = s.t.bytecode;
  if (ix.tab.n_rows == 0) return 0;
  u32 r = 0;
  int n;
  if (s.pos_mode == 1 || (pos_enabled(ix) && ix.pos_kind == ZK_POS_RUNS)) {
    Fr got;
    n = s.narrow == 1 ? pos_lookup_run<true>(ix, key, n_head, head, run_len, &r, live, B_VALUE, &got)
                      : pos_lookup_run<false>(ix, key, n_head, head, run_len, &r, live, B_VALUE, &got);
    if (live && n == 1) *value = got;
    return n;
  } else {
    Fr h = fr_add(h0, rlc_term(ix, key[2], 2));
    h = fr_add(h, rlc_term(ix, key[3], 3));
    h = fr_add(h, rlc_term(ix, key[4], 4));
    n = probe_hashed<5>(ix, h, key, &r, s.mask, live);
  }
  if (live && n == 1) *value = table_cell(ix.tab, B_VALUE, r);
  return n;
}
// heads-index probe of the step's code hash (no-op unless the bytecode table is positional)
ZK_HD int bytecode_head(const StepCtx& s, bool live, const Fr& hlo, const Fr& hhi, u32* head, u32* run_len) {
  const IndexDev& ix = s.t.bytecode;
  *head = 0;
  *run_len = 0;
  if (s.pos_mode != 1 && (ix.tab.n_rows == 0 || !(pos_enabled(ix) && ix.pos_kind == ZK_POS_RUNS))) return 0;
  return heads_probe(ix, hlo, hhi, head, run_len, s.mask, live);
}
// constant terms of a stack lookup's key hash, computed once per thread
ZK_HD void stack_key_pre(const IndexDev& rw_ix, Fr out[2]) {
  const Fr tag_term = rlc_term(rw_ix, fr_u64(ZK_TARGET_Stack), 2);
  out[0] = tag_term;
  out[1] = fr_add(rlc_term(rw_ix, fr_u64(1), 1), tag_term);
}
ZK_HD int rw_lookup(const StepCtx& s, bool live, const Fr& rwc, u64 rw, u64 tag, const Fr& id, const Fr& addr,
                    Word2* value) {
  Fr key[5] = {rwc, fr_u64(rw), fr_u64(tag), id, addr};
  u32 r;
  int n = 0;
  const IndexDev& ix = s.t.rw;
  if (s.pos_mode == 1 || (ix.tab.n_rows != 0 && pos_enabled(ix) && ix.pos_kind == ZK_POS_DENSE)) {
    Fr lo, hi;
    n = s.narrow == 1 ? pos_lookup_dense<5, true>(ix, key, &r, live, s.rw_base, R_VAL_LO, &lo, R_VAL_HI, &hi)
                      : pos_lookup_dense<5, false>(ix, key, &r, live, s.rw_base, R_VAL_LO, &lo, R_VAL_HI, &hi);
    if (live && n == 1) {
      value->lo = lo;
      value->hi = hi;
    }
    return n;
  } else if (ix.tab.n_rows != 0) {
    Fr h;
    if (tag == ZK_TARGET_Stack && s.stack_pre) {
      h = fr_add(fr_add(rwc, s.stack_pre[rw & 1]), fr_add(rlc_term(ix, id, 3), rlc_term(ix, addr, 4)));
    } else {
      h = rlc_key<5>(ix, key);
    }
    n = probe_hashed<5>(ix, h, key, &r, s.mask, live);
  }
  if (live && n == 1) {
    value->lo = table_cell(s.t.rw.tab, R_VAL_LO, r);
    value->hi = table_cell(s.t.rw.tab, R_VAL_HI, r);
  }
  return n;
}

// ---- prologue: verify_step before the gadget (main.py:47-63, instruction.py:189-204) --------
// Steps are bucketed by execution state (one bucket per state; the MUL state is split three ways by an
// opcode peek, see k_evm_classify) and each bucket is run by the kernel of its gate-program group.
#define ZK_EVM_NB 128      // bucket ids: execution states 0..ZK_ES_COUNT-1, then
#define ZK_BK_DIV ZK_ES_COUNT        // MUL-state steps whose opcode peeks as DIV
#define ZK_BK_MOD (ZK_ES_COUNT + 1)  // ... as MOD (everything else stays in bucket ZK_ES_MUL)
#define ZK_BK_NONE 0xFF              // the step already failed in the prologue
// returns the execution state whose gate program must run for this step, or -1 if the step already failed
ZK_HD int step_prologue(const StepCtx& s, u32 flags) {
  const Fr cs = s.cur(S_STATE), ns = s.nxt(S_STATE);
  const bool is_first = (flags & ZK_FLAG_EVM_FIRST_STEP) && s.row == 0;
  const bool is_last = (flags & ZK_FLAG_EVM_LAST_STEP) && s.i == s.w.n_rows - 2;
  const bool cs_small = fr_fits64(cs) && cs.l[0] < ZK_ES_COUNT;
  if (is_first) {
    EV_CHECK_RET(EV_FIRST_STATE, fr_eq_u64(cs, ZK_ES_BeginTx) || fr_eq_u64(cs, ZK_ES_EndBlock), -1);
    EV_CHECK_RET(EV_FIRST_RWC, fr_eq_u64(s.cur(S_RWC), 1), -1);
  }
  if (is_last) {
    EV_CHECK_RET(EV_LAST_STATE, fr_eq_u64(cs, ZK_ES_EndBlock), -1);
  } else {
    if (fr_eq_u64(cs, ZK_ES_EndTx))
      EV_CHECK_RET(EV_TRANS_FROM_ENDTX, fr_eq_u64(ns, ZK_ES_BeginTx) || fr_eq_u64(ns, ZK_ES_EndBlock), -1);
    else if (fr_eq_u64(cs, ZK_ES_EndBlock))
      EV_CHECK_RET(EV_TRANS_FROM_ENDBLOCK, fr_eq_u64(ns, ZK_ES_EndBlock), -1);
    if (fr_eq_u64(ns, ZK_ES_BeginTx))
      EV_CHECK_RET(EV_TRANS_TO_BEGINTX, fr_eq_u64(cs, ZK_ES_EndTx), -1);
    else if (fr_eq_u64(ns, ZK_ES_EndTx))
      EV_CHECK_RET(EV_TRANS_TO_ENDTX, (cs_small && ES_HALTS(cs.l[0])) || fr_eq_u64(cs, ZK_ES_BeginTx), -1);
    else if (fr_eq_u64(ns, ZK_ES_EndBlock))
      EV_CHECK_RET(EV_TRANS_TO_ENDBLOCK, fr_eq_u64(cs, ZK_ES_EndTx) || fr_eq_u64(cs, ZK_ES_EndBlock), -1);
  }
  EV_CHECK_RET(EV_NOT_IMPLEMENTED, cs_small && ES_IMPL(cs.l[0]), -1);
  if (ES_BUILT(cs.l[0])) return (int)cs.l[0];
  step_fail(s, EV_UNSUPPORTED_STATE);
  return -1;
}

// opcode_lookup(True) at the start of every hot gadget (instruction.py:784-790)
ZK_HD bool opcode_lookup(const StepCtx& s, bool live, Fr* opcode) {
  return need1(s, live, bytecode_lookup(s, live, s.cur(S_HASH_LO), s.cur(S_HASH_HI), 2, s.cur(S_PC), 1, opcode),
               EV_OP_UNSAT);
}

// responsible_opcode_lookup (instruction.py:779-782): fixed_table contains (13, state, opcode, 0)
ZK_HD bool responsible_opcode(const StepCtx& s, const Fr& state, const Fr& opcode) {
  if (fr_fits64(state) && state.l[0] < 256 && fr_fits64(opcode) && opcode.l[0] < 256) {
    const u32 bit = (u32)(state.l[0] << 8 | opcode.l[0]);
    return (s.resp[bit >> 5] >> (bit & 31)) & 1;
  }
  Fr key[4] = {fr_u64(ZK_FIXED_ResponsibleOpcode), state, opcode, fr_u64(0)};
  u32 r;
  return lookup<4>(s.t.fixed, key, &r) >= 1;  // out-of-range query: exact probe of the hash index
}

// step_state_transition_in_same_context, instruction.py:365-394.  General form: the rw_counter
// delta is a field element, memory_word_size either stays or moves To a value, and a dynamic gas
// cost is added to the opcode's constant cost.
ZK_HD void same_context_x(const StepCtx& s, const Fr& opcode, const Fr& d_rwc, const Fr& d_pc, const Fr& d_sp,
                          bool mem_to, const Fr& mem_value, const Fr& dyn_gas, u64 d_rev = 0, const Fr* d_log = nullptr) {
  EV_CHECK(EV_SC_RESP_OPCODE, responsible_opcode(s, s.cur(S_STATE), opcode));
  int gas_cost = -1;
  if (fr_fits64(opcode) && opcode.l[0] < 256) gas_cost = OPCODE_GAS(opcode.l[0]);
  EV_CHECK(EV_SC_OPCODE_VALUE, gas_cost >= 0);
  const Fr gas_after = fr_sub(s.cur(S_GAS), fr_add_u64(dyn_gas, (u64)gas_cost));
  EV_CHECK(EV_SC_GAS_RANGE, fr_fits64(gas_after));
  EV_CHECK(EV_SC_RWC, fr_eq(s.nxt(S_RWC), fr_add(s.cur(S_RWC), d_rwc)));
  EV_CHECK(EV_SC_PC, fr_eq(s.nxt(S_PC), fr_add(s.cur(S_PC), d_pc)));
  EV_CHECK(EV_SC_SP, fr_eq(s.nxt(S_SP), fr_add(s.cur(S_SP), d_sp)));
  EV_CHECK(EV_SC_GAS, fr_eq(s.nxt(S_GAS), gas_after));
  EV_CHECK(EV_SC_MEM, fr_eq(s.nxt(S_MEM), mem_to ? mem_value : s.cur(S_MEM)));
  EV_CHECK(EV_SC_REV, fr_eq(s.nxt(S_REV), d_rev ? fr_add_u64(s.cur(S_REV), d_rev) : s.cur(S_REV)));
  EV_CHECK(EV_SC_LOG, fr_eq(s.nxt(S_LOG), d_log ? fr_add(s.cur(S_LOG), *d_log) : s.cur(S_LOG)));
  EV_CHECK(EV_SC_CALL_ID, fr_eq(s.nxt(S_CALL_ID), s.cur(S_CALL_ID)));
  EV_CHECK(EV_SC_IS_ROOT, fr_eq(s.nxt(S_IS_ROOT), s.cur(S_IS_ROOT)));
  EV_CHECK(EV_SC_IS_CREATE, fr_eq(s.nxt(S_IS_CREATE), s.cur(S_IS_CREATE)));
  EV_CHECK(EV_SC_CODE_HASH,
           fr_eq(s.nxt(S_HASH_LO), s.cur(S_HASH_LO)) && fr_eq(s.nxt(S_HASH_HI), s.cur(S_HASH_HI)));
}
ZK_HD void same_context(const StepCtx& s, const Fr& opcode, u64 d_rwc, const Fr& d_pc, const Fr& d_sp) {
  same_context_x(s, opcode, fr_u64(d_rwc), d_pc, d_sp, false, fr_u64(0), fr_u64(0));
}

// add_words([x, y]) with the final carry dropped (util/arithmetic.py:236-242)
ZK_HD Word2 add_words2(const Word2& x, const Word2& y) {
  const Fr slo = fr_add(x.lo, y.lo);
  const Fr shi = fr_add(fr_add(x.hi, y.hi), fr_u128(slo.l[2], slo.l[3]));
  return Word2{fr_u128(slo.l[0], slo.l[1]), fr_u128(shi.l[0], shi.l[1])};
}

ZK_HD void gadget_add(const StepCtx& s, bool live) {
  Fr opcode = fr_u64(0);
  live = opcode_lookup(s, live, &opcode);
  const Fr rwc = s.cur(S_RWC), call_id = s.cur(S_CALL_ID), sp = s.cur(S_SP);
  const Fr sp1 = fr_add_u64(sp, 1);
  const Word2 zero{fr_u64(0), fr_u64(0)};
  Word2 a = zero, b = zero, c = zero;
  live = need1(s, live, rw_lookup(s, live, rwc, 0, ZK_TARGET_Stack, call_id, sp, &a), EV_ADD_A_UNSAT);
  live = need1(s, live, rw_lookup(s, live, fr_add_u64(rwc, 1), 0, ZK_TARGET_Stack, call_id, sp1, &b), EV_ADD_B_UNSAT);
  live = need1(s, live, rw_lookup(s, live, fr_add_u64(rwc, 2), 1, ZK_TARGET_Stack, call_id, sp1, &c), EV_ADD_C_UNSAT);
  if (!live) return;  // past the last lookup: plain early exits from here on
  const bool is_sub = fr_eq_u64(opcode, 3);
  EV_CHECK(EV_ADD_SUM, word_eq(add_words2(is_sub ? c : a, b), is_sub ? a : c));
  same_context(s, opcode, 3, fr_u64(1), fr_u64(1));
}

// ---- 256/512-bit integer helpers for the witness assignment of mul_div_mod.py:23-41 ----
ZK_HD void word_to_u256(const Word2& w, u64 o[4]) {
  o[0] = w.lo.l[0]; o[1] = w.lo.l[1]; o[2] = w.hi.l[0]; o[3] = w.hi.l[1];
}
ZK_HD Word2 u256_to_word(const u64 v[4]) {
  return Word2{fr_u128(v[0], v[1]), fr_u128(v[2], v[3])};
}
ZK_HD int cmp256(const u64 a[4], const u64 b[4]) {
#pragma unroll
  for (int k = 3; k >= 0; k--) {
    if (a[k] < b[k]) return -1;
    if (a[k] > b[k]) return 1;
  }
  return 0;
}
ZK_HD void sub256(const u64 a[4], const u64 b[4], u64 o[4]) {
  u64 br = 0;
#pragma unroll
  for (int k = 0; k < 4; k++) o[k] = sbb64(a[k], b[k], br);
}
// true iff b*a > d as integers (i.e. d - b*a < 0)
ZK_HD bool mul256_exceeds(const u64 a[4], const u64 b[4], const u64 d[4], u64 prod_lo[4]) {
  u64 t[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
  for (int x = 0; x < 4; x++) {
    u64 c = 0;
#pragma unroll
    for (int y = 0; y < 4; y++) {
      unsigned __int128 v = (unsigned __int128)a[x] * b[y] + t[x + y] + c;
      t[x + y] = (u64)v;
      c = (u64)(v >> 64);
    }
    t[x + 4] = c;
  }
#pragma unroll
  for (int k = 0; k < 4; k++) prod_lo[k] = t[k];
  return (t[4] | t[5] | t[6] | t[7]) != 0 || cmp256(prod_lo, d) > 0;
}
ZK_HD int bitlen256(const u64 v[4]) {
#ifdef __CUDA_ARCH__
#define ZK_CLZ64(x) __clzll((long long)(x))
#else
#define ZK_CLZ64(x) __builtin_clzll(x)
#endif
  if (v[3]) return 256 - ZK_CLZ64(v[3]);
  if (v[2]) return 192 - ZK_CLZ64(v[2]);
  if (v[1]) return 128 - ZK_CLZ64(v[1]);
  if (v[0]) return 64 - ZK_CLZ64(v[0]);
  return 0;
}
// (u1:u0) / v for a normalised v (bit 63 set) and u1 < v: two 64/32 steps (Hacker's Delight divlu)
ZK_HD u64 div128by64(u64 u1, u64 u0, u64 v) {
  const u64 b = 1ull << 32, vn1 = v >> 32, vn0 = v & 0xFFFFFFFFull, un1 = u0 >> 32, un0 = u0 & 0xFFFFFFFFull;
  u64 q1 = u1 / vn1, rhat = u1 - q1 * vn1;
  while (q1 >= b || q1 * vn0 > ((rhat << 32) | un1)) {
    q1--;
    rhat += vn1;
    if (rhat >= b) break;
  }
  const u64 un21 = ((u1 << 32) | un1) - q1 * v;  // mod 2^64, exact
  u64 q0 = un21 / vn1;
  rhat = un21 - q0 * vn1;
  while (q0 >= b || q0 * vn0 > ((rhat << 32) | un0)) {
    q0--;
    rhat += vn1;
    if (rhat >= b) break;
  }
  return (q1 << 32) | q0;
}
// q = n / d for d != 0 (only MOD steps pay for it).  Knuth's algorithm D with 64-bit digits on
// operands shifted so that the divisor's top bit is bit 255: always 4 quotient digits, static limb
// indices, no data-dependent trip count — so the lanes of a warp stay together (the bit-serial
// shift-subtract it replaces ran up to 256 iterations in the slowest lane: profiles/README.md v20).
ZK_HD void div256(const u64 n[4], const u64 d[4], u64 q[4]) {
  q[0] = q[1] = q[2] = q[3] = 0;
  if (cmp256(n, d) < 0) return;
  const int sd = 256 - bitlen256(d);  // 0..255
  const int ws = sd >> 6, bs = sd & 63;
  // D = d << sd (top bit set), N = n << sd (8 limbs)
  u64 t[8], dd[4];
#pragma unroll
  for (int k = 0; k < 8; k++) {
    u64 v = 0;
#pragma unroll
    for (int w = 0; w < 4; w++)
      if (ws == w && k - w >= 0 && k - w < 4) v = n[k - w];
    t[k] = v;
  }
#pragma unroll
  for (int k = 0; k < 4; k++) {
    u64 v = 0;
#pragma unroll
    for (int w = 0; w < 4; w++)
      if (ws == w && k - w >= 0) v = d[k - w];
    dd[k] = v;
  }
  u64 N[8], D[4];
#pragma unroll
  for (int k = 7; k >= 0; k--) N[k] = bs ? ((t[k] << bs) | (k ? t[k - 1] >> (64 - bs) : 0)) : t[k];
#pragma unroll
  for (int k = 3; k >= 0; k--) D[k] = bs ? ((dd[k] << bs) | (k ? dd[k - 1] >> (64 - bs) : 0)) : dd[k];
  u64 r0 = N[4], r1 = N[5], r2 = N[6], r3 = N[7];  // running remainder < D
#pragma unroll
  for (int j = 3; j >= 0; j--) {
    // (r3 r2 r1 r0 N[j]) / D: estimate from the top two digits, then multiply-subtract and add back
    u64 qh = r3 >= D[3] ? ~0ull : div128by64(r3, r2, D[3]);
    u64 p[5], c = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const unsigned __int128 v = (unsigned __int128)qh * D[k] + c;
      p[k] = (u64)v;
      c = (u64)(v >> 64);
    }
    p[4] = c;
    u64 br = 0;
    u64 s0 = sbb64(N[j], p[0], br), s1 = sbb64(r0, p[1], br), s2 = sbb64(r1, p[2], br), s3 = sbb64(r2, p[3], br),
        s4 = sbb64(r3, p[4], br);
    bool neg = br != 0;
#pragma unroll
    for (int fix = 0; fix < 2; fix++) {  // the estimate is at most 2 too large
      if (neg) {
        u64 cy = 0;
        s0 = adc64(s0, D[0], cy);
        s1 = adc64(s1, D[1], cy);
        s2 = adc64(s2, D[2], cy);
        s3 = adc64(s3, D[3], cy);
        s4 = adc64(s4, 0, cy);
        qh--;
        if (cy) neg = false;
      }
    }
    q[j] = qh;
    r0 = s0;
    r1 = s1;
    r2 = s2;
    r3 = s3;
  }
}

// Word((sel*lo, sel*hi)) with the constructor's < 2^128 assertion (arithmetic.py:110-114)
ZK_HD bool word_select(const Word2& w, const Fr& sel, Word2* out) {
  if (fr_is_zero(sel)) {
    out->lo = out->hi = fr_u64(0);
    return true;
  }
  if (fr_eq_u64(sel, 1)) {
    *out = w;
    return word_in_domain(w);
  }
  const Fr sm = fr_to_mont(sel);
  out->lo = fr_montmul(sm, w.lo);
  out->hi = fr_montmul(sm, w.hi);
  return word_in_domain(*out);
}

// low 256 bits of a * b
ZK_HD void mul256_lo(const u64 a[4], const u64 b[4], u64 o[4]) {
  u64 t[4] = {0, 0, 0, 0};
#pragma unroll
  for (int x = 0; x < 4; x++) {
    u64 c = 0;
#pragma unroll
    for (int y = 0; y + x < 4; y++) {
      unsigned __int128 v = (unsigned __int128)a[x] * b[y] + t[x + y] + c;
      t[x + y] = (u64)v;
      c = (u64)(v >> 64);
    }
  }
#pragma unroll
  for (int k = 0; k < 4; k++) o[k] = t[k];
}
// MUL / DIV / MOD decided as a whole for stack words in the halves domain: true iff every constraint of
// mul_div_mod.py:23-64 holds.  In that domain the gate a * b + c == d (+ the 9-byte carries, overflow == 0 for
// DIV / MOD), the select equation and remainder < divisor are statements about 256-bit integers:
//   MUL  pop1 * pop2 == push (mod 2^256)
//   DIV  push * pop2 <= pop1 and pop1 - push * pop2 < pop2       (pop2 == 0: push == 0)
//   MOD  push < pop2, push <= pop1 and pop2 | pop1 - push         (pop2 == 0: push == 0)
// On false the caller runs the gate program proper, which names the failing constraint.
ZK_HD bool mul_fast_ok(u64 op, const Word2& pop1, const Word2& pop2, const Word2& push) {
  u64 p1[4], p2[4], ps[4], pl[4];
  word_to_u256(pop1, p1);
  word_to_u256(pop2, p2);
  word_to_u256(push, ps);
  if (op == 2) {
    mul256_lo(p1, p2, pl);
    return cmp256(pl, ps) == 0;
  }
  if ((p2[0] | p2[1] | p2[2] | p2[3]) == 0) return (ps[0] | ps[1] | ps[2] | ps[3]) == 0;
  if (op == 4) {
    if (mul256_exceeds(ps, p2, p1, pl)) return false;
    u64 c[4];
    sub256(p1, pl, c);
    return cmp256(c, p2) < 0;
  }
  if (cmp256(ps, p2) >= 0 || cmp256(p1, ps) < 0) return false;
  u64 t[4], q[4];
  sub256(p1, ps, t);
  div256(t, p2, q);
  if (mul256_exceeds(q, p2, t, pl)) return false;
  return cmp256(pl, t) == 0;
}
// the gate program proper, after the three stack lookups; true iff no constraint failed
ZK_HD_NOINLINE bool gadget_mul_exact(const StepCtx& s, const Fr& opcode, const Word2& pop1, const Word2& pop2, const Word2& push) {
  const Fr one = fr_u64(1);
  // mul_div_mod.py:14-16 (Lagrange selectors over the field)
  Fr is_mul, is_div, is_mod;
  if (fr_eq_u64(opcode, 2)) { is_mul = one; is_div = fr_u64(0); is_mod = fr_u64(0); }
  else if (fr_eq_u64(opcode, 4)) { is_mul = fr_u64(0); is_div = one; is_mod = fr_u64(0); }
  else if (fr_eq_u64(opcode, 6)) { is_mul = fr_u64(0); is_div = fr_u64(0); is_mod = one; }
  else {
    const Fr o2 = fr_sub(opcode, fr_u64(2)), o4 = fr_sub(opcode, fr_u64(4));
    const Fr f4 = fr_sub(fr_u64(4), opcode), f6 = fr_sub(fr_u64(6), opcode);
    is_mul = fr_montmul(fr_mul(f4, f6), ZK_MONT_INV8);
    is_div = fr_montmul(fr_mul(o2, f6), ZK_MONT_INV4);
    is_mod = fr_montmul(fr_mul(o2, o4), ZK_MONT_INV8);
  }
  const Word2 zero{fr_u64(0), fr_u64(0)};
  const bool in_domain = word_in_domain(pop1) && word_in_domain(pop2) && word_in_domain(push);
  // witness assignment by branch, mul_div_mod.py:23-41 (Python int arithmetic)
  Word2 a, b, c, d;
  if (fr_eq_u64(is_mul, 1)) {
    a = pop1; b = pop2; c = zero; d = push;
  } else {
    EV_CHECK_RET(EV_MUL_WITNESS_DOMAIN, in_domain, false);  // would need > 512-bit integers
    d = pop1; b = pop2;
    u64 dv[4], bv[4];
    word_to_u256(d, dv);
    word_to_u256(b, bv);
    if (fr_eq_u64(is_div, 1)) {
      a = push;
      u64 av[4], pl[4], cv[4];
      word_to_u256(a, av);
      EV_CHECK_RET(EV_MUL_WITNESS_NEG, !mul256_exceeds(av, bv, dv, pl), false);  // Word(d - b*a) with d < b*a
      sub256(dv, pl, cv);
      c = u256_to_word(cv);
    } else if ((bv[0] | bv[1] | bv[2] | bv[3]) == 0) {
      c = d; a = zero;
    } else {
      c = push;
      u64 cv[4], tv[4], qv[4];
      word_to_u256(c, cv);
      EV_CHECK_RET(EV_MUL_WITNESS_NEG, cmp256(dv, cv) >= 0, false);  // (d - c) // b < 0
      sub256(dv, cv, tv);
      div256(tv, bv, qv);
      a = u256_to_word(qv);
    }
  }
  const bool b_zero = fr_is_zero(fr_add(b.lo, b.hi));  // is_zero_word: field sum of the halves
  // mul_add_words, instruction.py:599-632
  EV_CHECK_RET(EV_MUL_TO64, word_in_domain(a) && word_in_domain(b), false);
  Fr carry_lo, carry_hi, overflow;
  mul_add_carries(a, b, c, d, &carry_lo, &carry_hi, &overflow);
  EV_CHECK_RET(EV_MUL_CARRY_LO, fits_9_bytes(carry_lo), false);  // range_check(.., 9)
  EV_CHECK_RET(EV_MUL_CARRY_HI, fits_9_bytes(carry_hi), false);
  // the two constrain_equal of instruction.py:629-630 hold by construction of the carries
  // mul_div_mod.py:47-54: select_word's bool assert, then Word range asserts of select / +
  const bool mul0 = fr_is_zero(is_mul), mul1 = fr_eq_u64(is_mul, 1);
  EV_CHECK_RET(EV_MUL_SELECT, mul0 || mul1, false);
  Word2 t_d, t_a, t_c, sum;
  const Fr sel_a = b_zero ? fr_u64(0) : is_div, sel_c = b_zero ? fr_u64(0) : is_mod;
  EV_CHECK_RET(EV_MUL_SELECT, word_select(d, is_mul, &t_d) && word_select(a, sel_a, &t_a), false);
  EV_CHECK_RET(EV_MUL_SELECT, word_select(c, sel_c, &t_c), false);
  sum.lo = fr_add(t_d.lo, t_a.lo);
  sum.hi = fr_add(t_d.hi, t_a.hi);
  EV_CHECK_RET(EV_MUL_SELECT, word_in_domain(sum), false);
  sum.lo = fr_add(sum.lo, t_c.lo);
  sum.hi = fr_add(sum.hi, t_c.hi);
  EV_CHECK_RET(EV_MUL_SELECT, word_in_domain(sum), false);
  EV_CHECK_RET(EV_MUL_PUSH_EQ, word_eq(push, sum), false);
  // :57  is_mul * sum(c.to_le_bytes()) == 0  (is_mul is 0/1 here; byte sum < p)
  EV_CHECK_RET(EV_MUL_C_ZERO, mul0 || (fr_is_zero(c.lo) && fr_is_zero(c.hi)), false);
  // :60-61  (1-is_mul)*(1-b0)*(1-lt) == 0 with lt = compare_word(c, b)
  const bool lt = fr_lt(c.hi, b.hi) || (fr_eq(c.hi, b.hi) && fr_lt(c.lo, b.lo));
  EV_CHECK_RET(EV_MUL_REM_LT, mul1 || b_zero || lt, false);
  EV_CHECK_RET(EV_MUL_OVERFLOW, mul1 || fr_is_zero(overflow), false);
  return true;
}
ZK_HD void gadget_mul(const StepCtx& s, bool live) {
  Fr opcode = fr_u64(0);
  live = opcode_lookup(s, live, &opcode);
  const Fr rwc = s.cur(S_RWC), call_id = s.cur(S_CALL_ID), sp = s.cur(S_SP);
  const Fr sp1 = fr_add_u64(sp, 1);
  const Fr one = fr_u64(1);
  const Word2 zero{fr_u64(0), fr_u64(0)};
  Word2 pop1 = zero, pop2 = zero, push = zero;
  live = need1(s, live, rw_lookup(s, live, rwc, 0, ZK_TARGET_Stack, call_id, sp, &pop1), EV_MUL_POP1_UNSAT);
  live = need1(s, live, rw_lookup(s, live, fr_add_u64(rwc, 1), 0, ZK_TARGET_Stack, call_id, sp1, &pop2), EV_MUL_POP2_UNSAT);
  live = need1(s, live, rw_lookup(s, live, fr_add_u64(rwc, 2), 1, ZK_TARGET_Stack, call_id, sp1, &push), EV_MUL_PUSH_UNSAT);
  if (!live) return;  // past the last lookup: plain early exits from here on
  // the whole step decided at once when the words are in the halves domain and the opcode is one of the three;
  // anything else (and every failing step) runs the gate program proper.  Copies go to the out-of-line call so
  // that the passing path keeps its operands in registers.
  const bool in_dom = word_in_domain(pop1) && word_in_domain(pop2) && word_in_domain(push);
  const bool op_ok = fr_fits64(opcode) && (opcode.l[0] == 2 || opcode.l[0] == 4 || opcode.l[0] == 6);
  if (!(in_dom && op_ok && mul_fast_ok(opcode.l[0], pop1, pop2, push))) {
    const Fr o2 = opcode;
    const Word2 a2 = pop1, b2 = pop2, c2 = push;
    if (!gadget_mul_exact(s, o2, a2, b2, c2)) return;
  }
  same_context(s, opcode, 3, one, one);
}

// ---- PUSH (execution/push.py:6-33).  Generic (hash-index) form, written as lane functions: in
// k_evm_push_hash half a warp checks one PUSH step — sub-lane L owns pushed bytes L and L+16 (their
// bytecode lookups + equalities); tests/emu runs the same lane functions serially.  Positional tables
// take the thread-per-step form further down (gadget_push_pos1).
struct PushCommon {
  Fr hlo, hhi, h0, pc, opcode, num_pushed;
  int n_head;  // heads-index probe of the code hash (positional bytecode table)
  u32 run_len;  // Byte rows of that contract's run
  u32 head;
  u64 n_push, n_pad;
  Word2 value;
};
// program order up to the byte loop: opcode lookup, bytecode_length lookup, compare() range
// asserts, stack_push lookup, to_le_bytes(); false if the step failed (recorded if s.record)
ZK_HD bool push_prepare(const StepCtx& s, int n_op, const Fr& opcode, int n_len, const Fr& code_length,
                        int n_rw, const Word2& value, PushCommon* c) {
  if (!need1(s, true, n_op, EV_OP_UNSAT)) return false;
  if (!need1(s, true, n_len, EV_PUSH_LEN_UNSAT)) return false;
  c->opcode = opcode;
  c->num_pushed = fr_sub_u64(opcode, 0x5f);
  const Fr left = fr_sub_u64(fr_sub(code_length, c->pc), 1);
  EV_CHECK_RET(EV_PUSH_CMP_RANGE, fr_fits64(left) && fr_fits64(c->num_pushed), false);
  c->n_push = c->num_pushed.l[0];
  c->n_pad = left.l[0] < c->n_push ? c->n_push - left.l[0] : 0;
  if (!need1(s, true, n_rw, EV_PUSH_RW_UNSAT)) return false;
  EV_CHECK_RET(EV_PUSH_VALUE_BYTES, word_in_domain(value), false);
  c->value = value;
  return true;
}
// byte idx of the pushed word: returns the failing constraint id, or -1.  Warp-synchronous: every
// lane of s.mask calls it (the lookup inside is skipped with live = false where no byte is pushed)
ZK_HD int push_byte(const StepCtx& s, const PushCommon& c, int idx, bool live) {
  const u64 lo_limb = (idx & 8) ? c.value.lo.l[1] : c.value.lo.l[0];
  const u64 hi_limb = (idx & 8) ? c.value.hi.l[1] : c.value.hi.l[0];
  const u64 limb = idx < 16 ? lo_limb : hi_limb;
  const u64 byte = (limb >> (8 * (idx & 7))) & 0xFF;
  const int base = EV_PUSH_B0_UNSAT + 4 * idx;
  const bool pushed = live && (u64)idx < c.n_push && (u64)idx >= c.n_pad;
  Fr got = fr_u64(0);
  const Fr index = fr_sub_u64(fr_add(c.pc, c.num_pushed), (u64)idx);  // pc + num_pushed - idx
  const int n = bytecode_lookup_h(s, pushed, c.h0, c.n_head, c.head, c.run_len, c.hlo, c.hhi, 2, index, 0, &got);
  if (pushed) {
    if (n != 1) return n == 0 ? base : base + 1;
    return fr_eq_u64(got, byte) ? -1 : base + 2;
  }
  return byte == 0 ? -1 : base + 3;
}
ZK_HD void push_epilogue(const StepCtx& s, const PushCommon& c) {
  same_context(s, c.opcode, 1, fr_add_u64(c.num_pushed, 1), fr_sub(fr_u64(0), fr_u64(1)));
}
// The shared epilogue spread over a warp: lane c < 13 loads cell c of the current and next
// step and evaluates the transition constraint of that cell; returns the id of its failing
// constraint or INT_MAX.  Ids are in program order, so the warp minimum is the first failure.
ZK_HD int same_context_lane(const StepCtx& s, int lane, const Fr& cur, const Fr& nxt, const Fr& opcode, u64 d_rwc,
                            const Fr& d_pc, const Fr& d_sp) {
  const int kNone = 0x7FFFFFFF;
  if (lane >= 13) return kNone;
  int gas_cost = -1;
  if (fr_fits64(opcode) && opcode.l[0] < 256) gas_cost = OPCODE_GAS(opcode.l[0]);
  switch (lane) {
    case S_STATE:
      if (!responsible_opcode(s, cur, opcode)) return EV_SC_RESP_OPCODE;
      return gas_cost >= 0 ? kNone : EV_SC_OPCODE_VALUE;
    case S_GAS: {
      if (gas_cost < 0) return kNone;  // reported by lane S_STATE with a smaller id
      const Fr gas_after = fr_sub_u64(cur, (u64)gas_cost);
      if (!fr_fits64(gas_after)) return EV_SC_GAS_RANGE;
      return fr_eq(nxt, gas_after) ? kNone : EV_SC_GAS;
    }
    case S_RWC: return fr_eq(nxt, fr_add_u64(cur, d_rwc)) ? kNone : EV_SC_RWC;
    case S_PC: return fr_eq(nxt, fr_add(cur, d_pc)) ? kNone : EV_SC_PC;
    case S_SP: return fr_eq(nxt, fr_add(cur, d_sp)) ? kNone : EV_SC_SP;
    case S_MEM: return fr_eq(nxt, cur) ? kNone : EV_SC_MEM;
    case S_REV: return fr_eq(nxt, cur) ? kNone : EV_SC_REV;
    case S_LOG: return fr_eq(nxt, cur) ? kNone : EV_SC_LOG;
    case S_CALL_ID: return fr_eq(nxt, cur) ? kNone : EV_SC_CALL_ID;
    case S_IS_ROOT: return fr_eq(nxt, cur) ? kNone : EV_SC_IS_ROOT;
    case S_IS_CREATE: return fr_eq(nxt, cur) ? kNone : EV_SC_IS_CREATE;
    default: return fr_eq(nxt, cur) ? kNone : EV_SC_CODE_HASH;  // S_HASH_LO, S_HASH_HI
  }
}

// serial form (tests/emu, and any caller without a warp): s.mask names the calling thread only
ZK_HD void gadget_push(const StepCtx& s, bool live) {
  PushCommon c;
  c.hlo = s.cur(S_HASH_LO);
  c.hhi = s.cur(S_HASH_HI);
  c.pc = s.cur(S_PC);
  c.h0 = bytecode_hash0(s, c.hlo, c.hhi);
  Fr opcode = fr_u64(0), code_length = fr_u64(0);
  Word2 value{fr_u64(0), fr_u64(0)};
  c.n_head = bytecode_head(s, live, c.hlo, c.hhi, &c.head, &c.run_len);
  const int n_op = bytecode_lookup_h(s, live, c.h0, c.n_head, c.head, c.run_len, c.hlo, c.hhi, 2, c.pc, 1, &opcode);
  const int n_len = bytecode_lookup_h(s, live, c.h0, c.n_head, c.head, c.run_len, c.hlo, c.hhi, 1, fr_u64(0), 0, &code_length);
  const int n_rw = rw_lookup(s, live, s.cur(S_RWC), 1, ZK_TARGET_Stack, s.cur(S_CALL_ID), fr_sub_u64(s.cur(S_SP), 1), &value);
  if (!live) return;
  if (!push_prepare(s, n_op, opcode, n_len, code_length, n_rw, value, &c)) return;
  for (int idx = 0; idx < 32; idx++) {
    const int fid = push_byte(s, c, idx, true);
    if (fid >= 0) {
      step_fail(s, fid);
      return;
    }
  }
  push_epilogue(s, c);
}

// ---- PUSH on positional tables, ONE THREAD per step ------------------------------------------
// With positional rw + bytecode tables a PUSH step needs, per pushed byte, only the is_code and
// value cells of row head + 1 + index (lookup.cuh:pos_lookup_run): 64 narrow, independent loads of
// two columns.  One thread per step issues them back to back with no branch in between (the
// outcome of every byte is folded into three bit masks, the first set bit in program order names
// the failing constraint), so a warp instruction serves 32 steps instead of the 2 of the
// half-warp kernel below.  `hc` caches the heads-index probe of the last code hash this thread saw.
struct HeadCache {
  Fr hlo, hhi;
  u32 head, len;
  int n;
  bool have;
};
ZK_HD bool both_positional(const EvmTables& t) {
  return t.rw.tab.n_rows != 0 && t.bytecode.tab.n_rows != 0 && pos_enabled(t.rw) && pos_enabled(t.bytecode) &&
         t.rw.pos_kind == ZK_POS_DENSE && t.bytecode.pos_kind == ZK_POS_RUNS;
}
// the 32 byte lookups of a PUSH step as three bit masks (bit idx: lookup unsat / value differs / a
// non-pushed byte is not zero).  WIS / WVAL = compile-time widths of the is_code / value columns, or
// 0 for the generic loader.
template <int WIS, int WVAL>
ZK_HD void push_byte_masks(const TableDev& bt, const PushCommon& c, const Fr& top, bool top_ok, u32* m_unsat,
                           u32* m_neq, u32* m_pad) {
  const unsigned char* p_is = bt.base + bt.off[B_ISCODE];
  const unsigned char* p_val = bt.base + bt.off[B_VALUE];
  const u32 w_is = bt.width[B_ISCODE], w_val = bt.width[B_VALUE];
  const u64 first_row = (u64)c.head + 1;
  u32 mu = 0, mn = 0, mp = 0;
#pragma unroll
  for (int idx = 0; idx < 32; idx++) {
    const u64 lo_limb = (idx & 8) ? c.value.lo.l[1] : c.value.lo.l[0];
    const u64 hi_limb = (idx & 8) ? c.value.hi.l[1] : c.value.hi.l[0];
    const u64 byte = ((idx < 16 ? lo_limb : hi_limb) >> (8 * (idx & 7))) & 0xFF;
    const bool pushed = (u64)idx < c.n_push && (u64)idx >= c.n_pad;
    const bool valid = pushed && top_ok && top.l[0] >= (u64)idx && top.l[0] - (u64)idx < (u64)c.run_len;
    const u64 row = valid ? first_row + (top.l[0] - (u64)idx) : 0;
    const Fr is_code = WIS ? ld_col_c<WIS>(p_is, row) : ld_col(p_is, w_is, row);
    const Fr got = WVAL ? ld_col_c<WVAL>(p_val, row) : ld_col(p_val, w_val, row);
    const bool hit = valid && fr_is_zero(is_code);  // key: (hash, Byte, index, is_code = 0)
    mu |= (u32)(pushed && !hit) << idx;
    mn |= (u32)(hit && !fr_eq_u64(got, byte)) << idx;
    mp |= (u32)(!pushed && byte != 0) << idx;
  }
  *m_unsat = mu;
  *m_neq = mn;
  *m_pad = mp;
}
ZK_HD_NOINLINE void push_byte_masks_ni(const TableDev& bt, const PushCommon& c, const Fr& top, bool top_ok, u32* m_unsat, u32* m_neq,
                                       u32* m_pad) {
  push_byte_masks<0, 0>(bt, c, top, top_ok, m_unsat, m_neq, m_pad);
}
// The same 32 lookups decided all at once for the layout every packer produces (is_code 1 byte, value 4 bytes):
// true iff every one of them holds.  The rows of the pushed bytes are consecutive, downwards from index
// pc + num_pushed, so the loads are one base pointer each with compile-time offsets, predicated by a bit of the
// valid-index mask; the looked-up bytes are assembled into eight 32-bit words that must equal the pushed word
// (which also makes the non-pushed bytes zero).  On false the caller runs push_byte_masks to name the first
// failing constraint in program order — failing steps pay twice, passing steps ~6 instructions per byte.
ZK_HD u32 bits_below(u32 x) { return x >= 32 ? 0xFFFFFFFFu : (1u << x) - 1u; }
ZK_HD bool push_bytes_all_ok(const TableDev& bt, const PushCommon& c, const Fr& top, bool top_ok) {
  const u32 n_push = c.n_push < 32 ? (u32)c.n_push : 32u, n_pad = c.n_pad < 32 ? (u32)c.n_pad : 32u;
  const u32 pushed = n_push > n_pad ? (bits_below(n_push) & ~bits_below(n_pad)) : 0u;
  // valid idx: idx <= top and top - idx < run_len
  const u64 t = top.l[0];
  const u32 v_hi = t >= 31 ? 32u : (u32)t + 1u;
  const u64 below = t >= (u64)c.run_len ? t - (u64)c.run_len + 1 : 0;
  const u32 v_lo = below < 32 ? (u32)below : 32u;
  const u32 valid = top_ok ? (pushed & bits_below(v_hi) & ~bits_below(v_lo)) : 0u;
  if (pushed & ~valid) return false;  // a pushed byte without a row
  const u64 base_row = (u64)c.head + 1 + t;
  const unsigned char* q_is = bt.base + bt.off[B_ISCODE] + base_row;
  const u32* q_val = (const u32*)(bt.base + bt.off[B_VALUE]) + base_row;
  u32 acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  u32 is_any = 0, wide = 0;
#pragma unroll
  for (int idx = 0; idx < 32; idx++) {
    if ((valid >> idx) & 1) {
#ifdef __CUDA_ARCH__
      const u32 ic = __ldg(q_is - idx), g = __ldg(q_val - idx);
#else
      const u32 ic = q_is[-idx], g = q_val[-idx];
#endif
      is_any |= ic;
      wide |= g;
      acc[idx >> 2] |= g << (8 * (idx & 3));
    }
  }
  const u64 v0 = c.value.lo.l[0], v1 = c.value.lo.l[1], v2 = c.value.hi.l[0], v3 = c.value.hi.l[1];
  const u32 diff = (acc[0] ^ (u32)v0) | (acc[1] ^ (u32)(v0 >> 32)) | (acc[2] ^ (u32)v1) | (acc[3] ^ (u32)(v1 >> 32)) |
                   (acc[4] ^ (u32)v2) | (acc[5] ^ (u32)(v2 >> 32)) | (acc[6] ^ (u32)v3) | (acc[7] ^ (u32)(v3 >> 32));
  return (is_any | (wide >> 8) | diff) == 0;
}
ZK_HD void gadget_push_pos1(const StepCtx& s, HeadCache* hc) {
  PushCommon c;
  c.hlo = s.cur(S_HASH_LO);
  c.hhi = s.cur(S_HASH_HI);
  c.pc = s.cur(S_PC);
  c.h0 = fr_u64(0);
  if (!(hc->have && fr_eq(c.hlo, hc->hlo) && fr_eq(c.hhi, hc->hhi))) {
    hc->n = bytecode_head(s, true, c.hlo, c.hhi, &hc->head, &hc->len);
    hc->hlo = c.hlo;
    hc->hhi = c.hhi;
    hc->have = true;
  }
  c.n_head = hc->n;
  c.head = hc->head;
  c.run_len = hc->len;
  Fr opcode = fr_u64(0), code_length = fr_u64(0);
  Word2 value{fr_u64(0), fr_u64(0)};
  const int n_op = bytecode_lookup_h(s, true, c.h0, c.n_head, c.head, c.run_len, c.hlo, c.hhi, 2, c.pc, 1, &opcode);
  const int n_len = bytecode_lookup_h(s, true, c.h0, c.n_head, c.head, c.run_len, c.hlo, c.hhi, 1, fr_u64(0), 0, &code_length);
  const int n_rw = rw_lookup(s, true, s.cur(S_RWC), 1, ZK_TARGET_Stack, s.cur(S_CALL_ID), fr_sub_u64(s.cur(S_SP), 1), &value);
  if (!push_prepare(s, n_op, opcode, n_len, code_length, n_rw, value, &c)) return;
  // byte idx is looked up at index = pc + num_pushed - idx (push.py:24-31); as a field element it
  // only names a row when it is a small non-negative integer
  const Fr top = fr_add(c.pc, c.num_pushed);
  const bool top_ok = fr_fits64(top) && c.n_head == 1;
  const TableDev& bt = s.t.bytecode.tab;
  // the layout every packer produces for these two columns (is_code 1 byte, value 4 bytes: the Header
  // row holds the code length) is decided as a whole first; a failing step, or any other layout, goes through
  // the per-byte masks with the generic per-width loader (copies of the operands: the out-of-line call must not
  // pin `c` in local memory on the passing path)
  const bool typed = bt.width[B_ISCODE] == 1 && bt.width[B_VALUE] == 4;
  if (!(typed && push_bytes_all_ok(bt, c, top, top_ok))) {
    const PushCommon c2 = c;
    const Fr top2 = top;
    u32 m_unsat = 0, m_neq = 0, m_pad = 0;
    push_byte_masks_ni(bt, c2, top2, top_ok, &m_unsat, &m_neq, &m_pad);
    const u32 any = m_unsat | m_neq | m_pad;
    if (any) {
#ifdef __CUDA_ARCH__
      const int idx = __ffs(any) - 1;
#else
      const int idx = __builtin_ctz(any);
#endif
      const int base = EV_PUSH_B0_UNSAT + 4 * idx;
      step_fail(s, ((m_unsat >> idx) & 1) ? base : (((m_neq >> idx) & 1) ? base + 2 : base + 3));
      return;
    }
  }
  push_epilogue(s, c);
}

ZK_HD void gadget_pop(const StepCtx& s, bool live) {
  Fr opcode = fr_u64(0);
  live = opcode_lookup(s, live, &opcode);
  Word2 y{fr_u64(0), fr_u64(0)};
  live = need1(s, live, rw_lookup(s, live, s.cur(S_RWC), 0, ZK_TARGET_Stack, s.cur(S_CALL_ID), s.cur(S_SP), &y),
               EV_POP_RW_UNSAT);
  if (!live) return;
  same_context(s, opcode, 1, fr_u64(1), fr_u64(1));
}

// Out-of-line copies of the shared lookups / epilogue for the RARE gate programs below: k_evm_misc holds
// two dozen gate programs, and with every lookup inlined (hash path + positional path each) it took
// ptxas 140 s to compile; the hot kernels keep the inlined forms.
ZK_HD_NOINLINE int rw_lookup_ni(const StepCtx& s, bool live, const Fr& rwc, u64 rw, u64 tag, const Fr& id, const Fr& addr,
                                Word2* value) {
  return rw_lookup(s, live, rwc, rw, tag, id, addr, value);
}
ZK_HD_NOINLINE int bytecode_lookup_ni(const StepCtx& s, bool live, const Fr& hlo, const Fr& hhi, u64 tag, const Fr& index,
                                      u64 is_code, Fr* value) {
  return bytecode_lookup(s, live, hlo, hhi, tag, index, is_code, value);
}
ZK_HD_NOINLINE bool opcode_lookup_ni(const StepCtx& s, bool live, Fr* opcode) { return opcode_lookup(s, live, opcode); }
ZK_HD_NOINLINE void same_context_x_ni(const StepCtx& s, const Fr& opcode, const Fr& d_rwc, const Fr& d_pc, const Fr& d_sp,
                                      bool mem_to, const Fr& mem_value, const Fr& dyn_gas) {
  same_context_x(s, opcode, d_rwc, d_pc, d_sp, mem_to, mem_value, dyn_gas);
}
// + reversible_write_counter = Transition.delta(d_rev)
ZK_HD_NOINLINE void same_context_r_ni(const StepCtx& s, const Fr& opcode, const Fr& d_rwc, const Fr& d_pc, const Fr& d_sp,
                                      const Fr& dyn_gas, u64 d_rev) {
  same_context_x(s, opcode, d_rwc, d_pc, d_sp, false, fr_u64(0), dyn_gas, d_rev);
}
ZK_HD_NOINLINE void same_context_ni(const StepCtx& s, const Fr& opcode, u64 d_rwc, const Fr& d_pc, const Fr& d_sp) {
  same_context_x(s, opcode, fr_u64(d_rwc), d_pc, d_sp, false, fr_u64(0), fr_u64(0));
}

// ---- SHA3 (execution/sha3.py:6-55) and CALLDATACOPY (execution/calldatacopy.py:6-62) ----------
// word_to_fq(word, 5) (instruction.py:480-484): 0 ok, 1 = to_le_bytes OverflowError, 2 = raise
ZK_HD int word_to_fq5(const Word2& w, Fr* out) {
  if (!word_in_domain(w)) return 1;
  if ((w.lo.l[0] >> 40) || w.lo.l[1] || w.hi.l[0] || w.hi.l[1]) return 2;
  *out = fr_u64(w.lo.l[0]);
  return 0;
}
ZK_HD u64 memory_gas_cost(u64 size) { return size * size / 512 + 3 * size; }  // size < 2^32 (instruction.py:1129-1136)
// memory_expansion_dynamic_length + memory_copier_gas_cost (instruction.py:1157-1192): 0 ok, else
// 1 + index of the failing check in {MEMSIZE_RANGE, MAX_RANGE, WORDSIZE_RANGE, GASCOST_RANGE}
ZK_HD_NOINLINE int copier_gas(const StepCtx& s, u64 offset, u64 length, u64 per_word, Fr* next_mem, Fr* gas) {
  const u64 cd_size = (offset + length + 31) / 32;  // offset, length < 2^40
  if (cd_size >> 32) return 1;
  const Fr cur = s.cur(S_MEM);
  if (!(fr_fits64(cur) && (cur.l[0] >> 32) == 0)) return 2;
  const u64 nxt = cur.l[0] < cd_size ? cd_size : cur.l[0];
  const u64 expansion = memory_gas_cost(nxt) - memory_gas_cost(cur.l[0]);
  const u64 words = (length + 31) / 32;
  if (words >> 32) return 3;
  const unsigned __int128 g = (unsigned __int128)words * per_word + expansion;
  if ((u64)(g >> 64)) return 4;
  *next_mem = fr_u64(nxt);
  *gas = fr_u64((u64)g);
  return 0;
}
// copy_lookup (instruction.py:1361-1386, table.py:760-787); ids are values (hi half 0)
ZK_HD_NOINLINE int copy_lookup(const StepCtx& s, bool live, const Fr& src_id, u64 src_tag, const Fr& dst_id, u64 dst_tag,
                      const Fr& src_addr, const Fr& src_end, const Fr& dst_addr, const Fr& length, const Fr& rwc,
                      Fr* rwc_inc, Fr* rlc_acc) {
  Fr key[11] = {src_id, fr_u64(0), fr_u64(src_tag), dst_id, fr_u64(0), fr_u64(dst_tag), src_addr, src_end,
                dst_addr, length, rwc};
  u32 r;
  const int n = lookup_sync<11>(s.t.copy, key, &r, s.mask, live);
  if (live && n == 1) {
    *rlc_acc = table_cell(s.t.copy.tab, 11, r);
    *rwc_inc = table_cell(s.t.copy.tab, 13, r);
  }
  return n;
}
// call_context_lookup: rw row (rw_counter, Read, CallContext, call_id, address = field tag)
ZK_HD_NOINLINE int call_context(const StepCtx& s, bool live, const Fr& rwc, const Fr& call_id, u64 field_tag, Fr* value,
                       bool* is_word) {
  Fr key[5] = {rwc, fr_u64(0), fr_u64(ZK_TARGET_CallContext), call_id, fr_u64(field_tag)};
  u32 r;
  const int n = lookup_sync<5>(s.t.rw, key, &r, s.mask, live);
  if (live && n == 1) {
    *value = table_cell(s.t.rw.tab, R_VAL_LO, r);
    *is_word = s.t.rw.tab.flags && (s.t.rw.tab.flags[r] & 1);
  }
  return n;
}
#define EV_LIVE_CHECK(id, cond)   \
  do {                            \
    if (live && !(cond)) {        \
      step_fail(s, (id));         \
      live = false;               \
    }                             \
  } while (0)

ZK_HD_NOINLINE void gadget_sha3(const StepCtx& s, bool live) {
  Fr opcode = fr_u64(0);
  live = opcode_lookup_ni(s, live, &opcode);
  const Fr rwc = s.cur(S_RWC), call_id = s.cur(S_CALL_ID), sp = s.cur(S_SP);
  const Fr sp1 = fr_add_u64(sp, 1);
  const Word2 zero{fr_u64(0), fr_u64(0)};
  Word2 off_w = zero, size_w = zero, val_w = zero;
  live = need1(s, live, rw_lookup_ni(s, live, rwc, 0, ZK_TARGET_Stack, call_id, sp, &off_w), EV_SHA_OFF_UNSAT);
  live = need1(s, live, rw_lookup_ni(s, live, fr_add_u64(rwc, 1), 0, ZK_TARGET_Stack, call_id, sp1, &size_w), EV_SHA_SIZE_UNSAT);
  live = need1(s, live, rw_lookup_ni(s, live, fr_add_u64(rwc, 2), 1, ZK_TARGET_Stack, call_id, sp1, &val_w), EV_SHA_VAL_UNSAT);
  Fr length = fr_u64(0), offset = fr_u64(0);
  if (live) {
    int rc = word_to_fq5(size_w, &length);
    EV_LIVE_CHECK(rc == 1 ? EV_SHA_LEN_BYTES : EV_SHA_LEN_RANGE, rc == 0);
    if (live && !fr_is_zero(length)) {
      rc = word_to_fq5(off_w, &offset);
      EV_LIVE_CHECK(rc == 1 ? EV_SHA_OFF_BYTES : EV_SHA_OFF_RANGE, rc == 0);
    }
  }
  Fr rwc_inc = fr_u64(0), rlc_acc = fr_u64(0);
  {
    const bool go = live && !fr_is_zero(length);
    const int n = copy_lookup(s, go, call_id, ZK_COPY_Memory, call_id, ZK_COPY_RlcAcc, offset, fr_add(offset, length),
                              fr_u64(0), length, fr_add_u64(rwc, 3), &rwc_inc, &rlc_acc);
    if (go) live = need1(s, live, n, EV_SHA_COPY_UNSAT);
  }
  {
    Fr key[3] = {fr_u64(2), rlc_acc, length};  // keccak_lookup(length, rlc_acc), state_tag = Finalize
    u32 hit = 0;
    const int n = lookup_sync<3>(s.t.keccak, key, &hit, s.mask, live);
    live = need1(s, live, n, EV_SHA_KECCAK_UNSAT);
    if (live)
      EV_LIVE_CHECK(EV_SHA_HASH_EQ, fr_eq(table_cell(s.t.keccak.tab, 3, hit), val_w.lo) &&
                                        fr_eq(table_cell(s.t.keccak.tab, 4, hit), val_w.hi));
  }
  if (!live) return;  // past the last lookup
  Fr next_mem, gas;
  const int rc = copier_gas(s, offset.l[0], length.l[0], ZK_GAS_COST_COPY_SHA3, &next_mem, &gas);
  EV_CHECK(EV_SHA_MEMSIZE_RANGE + rc - 1, rc == 0);
  same_context_x_ni(s, opcode, fr_add_u64(rwc_inc, 3), fr_u64(1), fr_u64(1), true, next_mem, gas);
}

ZK_HD_NOINLINE void gadget_calldatacopy(const StepCtx& s, bool live) {
  Fr opcode = fr_u64(0);
  live = opcode_lookup_ni(s, live, &opcode);
  const Fr rwc = s.cur(S_RWC), call_id = s.cur(S_CALL_ID), sp = s.cur(S_SP);
  const Word2 zero{fr_u64(0), fr_u64(0)};
  Word2 moff_w = zero, doff_w = zero, len_w = zero;
  live = need1(s, live, rw_lookup_ni(s, live, rwc, 0, ZK_TARGET_Stack, call_id, sp, &moff_w), EV_CDC_MOFF_UNSAT);
  live = need1(s, live, rw_lookup_ni(s, live, fr_add_u64(rwc, 1), 0, ZK_TARGET_Stack, call_id, fr_add_u64(sp, 1), &doff_w), EV_CDC_DOFF_UNSAT);
  live = need1(s, live, rw_lookup_ni(s, live, fr_add_u64(rwc, 2), 0, ZK_TARGET_Stack, call_id, fr_add_u64(sp, 2), &len_w), EV_CDC_LEN_UNSAT);
  Fr length = fr_u64(0), moff = fr_u64(0), doff = fr_u64(0);
  if (live) {
    int rc = word_to_fq5(len_w, &length);
    EV_LIVE_CHECK(rc == 1 ? EV_CDC_LEN_BYTES : EV_CDC_LEN_RANGE, rc == 0);
    if (live && !fr_is_zero(length)) {
      rc = word_to_fq5(moff_w, &moff);
      EV_LIVE_CHECK(rc == 1 ? EV_CDC_MOFF_BYTES : EV_CDC_MOFF_RANGE, rc == 0);
    }
    if (live) {
      rc = word_to_fq5(doff_w, &doff);
      EV_LIVE_CHECK(rc == 1 ? EV_CDC_DOFF_BYTES : EV_CDC_DOFF_RANGE, rc == 0);
    }
  }
  const Fr is_root = s.cur(S_IS_ROOT);
  const bool root = !fr_is_zero(is_root);  // Python truthiness of StepState.is_root
  Fr src_id = fr_u64(0), cd_len = fr_u64(0), cd_off = fr_u64(0);
  bool w = false;
  live = need1(s, live, call_context(s, live, fr_add_u64(rwc, 3), call_id, root ? ZK_CC_TxId : ZK_CC_CallerId, &src_id, &w), EV_CDC_CC1_UNSAT);
  EV_LIVE_CHECK(EV_CDC_CC1_TYPE, !w);
  live = need1(s, live, call_context(s, live, fr_add_u64(rwc, 4), call_id, ZK_CC_CallDataLength, &cd_len, &w), EV_CDC_CC2_UNSAT);
  EV_LIVE_CHECK(EV_CDC_CC2_TYPE, !w);
  {
    const bool go = live && !root;
    const int n = call_context(s, go, fr_add_u64(rwc, 5), call_id, ZK_CC_CallDataOffset, &cd_off, &w);
    if (go) {
      live = need1(s, live, n, EV_CDC_CC3_UNSAT);
      EV_LIVE_CHECK(EV_CDC_CC3_TYPE, !w);
    }
  }
  const u64 k = root ? 5 : 6;
  Fr next_mem = fr_u64(0), gas = fr_u64(0);
  if (live) {
    const int rc = copier_gas(s, moff.l[0], length.l[0], ZK_GAS_COST_COPY, &next_mem, &gas);
    EV_LIVE_CHECK(EV_CDC_MEMSIZE_RANGE + rc - 1, rc == 0);
    EV_LIVE_CHECK(EV_CDC_SELECT_BOOL, fr_fits64(is_root) && is_root.l[0] <= 1);
  }
  Fr rwc_inc = fr_u64(0), unused = fr_u64(0);
  {
    const bool go = live && !fr_is_zero(length);
    const int n = copy_lookup(s, go, src_id, root ? ZK_COPY_TxCalldata : ZK_COPY_Memory, call_id, ZK_COPY_Memory,
                              fr_add(cd_off, doff), fr_add(cd_off, cd_len), moff, length, fr_add_u64(rwc, k), &rwc_inc, &unused);
    if (go) live = need1(s, live, n, EV_CDC_COPY_UNSAT);
  }
  if (!live) return;
  same_context_x_ni(s, opcode, fr_add_u64(rwc_inc, k), fr_u64(1), fr_u64(3), true, next_mem, gas);
}

// ---- STOP (execution/stop.py:7-51) ------------------------------------------------------------
// call_context_lookup_word: rw row (rw_counter, rw, CallContext, call_id, address = field tag)
ZK_HD_NOINLINE int call_context_w(const StepCtx& s, bool live, const Fr& rwc, u64 rw, const Fr& call_id, u64 field_tag,
                         Word2* value, bool* is_word) {
  Fr key[5] = {rwc, fr_u64(rw), fr_u64(ZK_TARGET_CallContext), call_id, fr_u64(field_tag)};
  u32 r;
  const int n = lookup_sync<5>(s.t.rw, key, &r, s.mask, live);
  if (live && n == 1) {
    value->lo = table_cell(s.t.rw.tab, R_VAL_LO, r);
    value->hi = table_cell(s.t.rw.tab, R_VAL_HI, r);
    *is_word = s.t.rw.tab.flags && (s.t.rw.tab.flags[r] & 1);
  }
  return n;
}
// step_state_transition_to_restored_context (instruction.py:293-363) with caller_id = None:
// rw_off = rw lookups the gadget already did; add_rev = the current state halts in success.
// Lookup k has ids EV_RST0_UNSAT + 3k (+1 ambiguous, +2 value type / written value).
// extra_delta: rw counters the step consumes without looking them up (the reverted writes of an error state).
// General form: the 12 lookups sit at rw_counter + look_off + k, the next rw_counter is rw_counter + delta12 + 12 (the two
// differ in return_revert.py's CREATE branch, whose rwc_delta forgets two lookups).
ZK_HD_NOINLINE void restore_context_f(const StepCtx& s, bool live, const Fr& look_off, const Fr& delta12, const Fr& ret_off,
                                      const Fr& ret_len, const Fr& gas_left, bool add_rev) {
  const u64 READ_TAGS[8] = {ZK_CC_IsRoot,       ZK_CC_IsCreate, ZK_CC_CodeHash,   ZK_CC_ProgramCounter,
                            ZK_CC_StackPointer, ZK_CC_GasLeft,  ZK_CC_MemorySize, ZK_CC_ReversibleWriteCounter};
  const u64 WRITE_TAGS[3] = {ZK_CC_LastCalleeId, ZK_CC_LastCalleeReturnDataOffset, ZK_CC_LastCalleeReturnDataLength};
  const Fr rwc = s.cur(S_RWC), call_id = s.cur(S_CALL_ID);
  const Fr lrwc = fr_add(rwc, look_off);
  const Word2 zero{fr_u64(0), fr_u64(0)};
  Word2 v = zero;
  bool w = false;
  live = need1(s, live, call_context_w(s, live, lrwc, 0, call_id, ZK_CC_CallerId, &v, &w), EV_RST0_UNSAT);
  EV_LIVE_CHECK(EV_RST0_CHECK, !w);
  const Fr caller_id = v.lo;
  Word2 vals[8];
  bool any_word = false;  // of the seven fields read through .value() (CodeHash is a word)
  for (int k = 0; k < 8; k++) {
    vals[k] = zero;
    bool wk = false;
    live = need1(s, live, call_context_w(s, live, fr_add_u64(lrwc, 1 + k), 0, caller_id, READ_TAGS[k], &vals[k], &wk),
                 EV_RST0_UNSAT + 3 * (1 + k));
    if (live && k != 2) any_word |= wk;
  }
  for (int k = 0; k < 3; k++) {
    const Fr expected = k == 0 ? call_id : (k == 1 ? ret_off : ret_len);
    live = need1(s, live, call_context_w(s, live, fr_add_u64(lrwc, 9 + k), 1, caller_id, WRITE_TAGS[k], &v, &w),
                 EV_RST0_UNSAT + 3 * (9 + k));
    EV_LIVE_CHECK(EV_RST0_UNSAT + 3 * (9 + k) + 2, !w && fr_eq(v.lo, expected));
  }
  if (!live) return;  // past the last lookup
  EV_CHECK(EV_RST_VALUE_TYPE, !any_word);
  EV_CHECK(EV_RST_RWC, fr_eq(s.nxt(S_RWC), fr_add_u64(fr_add(rwc, delta12), 12)));
  EV_CHECK(EV_RST_CALL_ID, fr_eq(s.nxt(S_CALL_ID), caller_id));
  EV_CHECK(EV_RST_IS_ROOT, fr_eq(s.nxt(S_IS_ROOT), vals[0].lo));
  EV_CHECK(EV_RST_IS_CREATE, fr_eq(s.nxt(S_IS_CREATE), vals[1].lo));
  EV_CHECK(EV_RST_CODE_HASH, fr_eq(s.nxt(S_HASH_LO), vals[2].lo) && fr_eq(s.nxt(S_HASH_HI), vals[2].hi));
  EV_CHECK(EV_RST_PC, fr_eq(s.nxt(S_PC), vals[3].lo));
  EV_CHECK(EV_RST_SP, fr_eq(s.nxt(S_SP), vals[4].lo));
  EV_CHECK(EV_RST_GAS, fr_eq(s.nxt(S_GAS), fr_add(vals[5].lo, gas_left)));
  EV_CHECK(EV_RST_MEM, fr_eq(s.nxt(S_MEM), vals[6].lo));
  EV_CHECK(EV_RST_REV, fr_eq(s.nxt(S_REV), add_rev ? fr_add(vals[7].lo, s.cur(S_REV)) : vals[7].lo));
}
ZK_HD void restore_context_x(const StepCtx& s, bool live, u64 rw_off, const Fr& ret_off, const Fr& ret_len, const Fr& gas_left,
                            bool add_rev, const Fr& extra_delta) {
  restore_context_f(s, live, fr_u64(rw_off), fr_add_u64(extra_delta, rw_off), ret_off, ret_len, gas_left, add_rev);
}
ZK_HD void restore_context(const StepCtx& s, bool live, u64 rw_off, const Fr& ret_off, const Fr& ret_len, const Fr& gas_left,
                          bool add_rev) {
  restore_context_x(s, live, rw_off, ret_off, ret_len, gas_left, add_rev, fr_u64(0));
}

ZK_HD_NOINLINE void gadget_stop(const StepCtx& s, bool live) {
  const Fr hlo = s.cur(S_HASH_LO), hhi = s.cur(S_HASH_HI), pc = s.cur(S_PC);
  Fr code_length = fr_u64(0);
  live = need1(s, live, bytecode_lookup_ni(s, live, hlo, hhi, 1, fr_u64(0), 0, &code_length), EV_STOP_LEN_UNSAT);
  EV_LIVE_CHECK(EV_STOP_CMP_RANGE, fr_fits64(code_length) && fr_fits64(pc));
  {
    // is_within_range = 1 - lt(code_length, pc) - eq(code_length, pc)  (stop.py:12-18)
    const bool go = live && code_length.l[0] > pc.l[0];
    Fr opcode = fr_u64(0);
    const int n = bytecode_lookup_ni(s, go, hlo, hhi, 2, pc, 1, &opcode);
    if (go) {
      live = need1(s, live, n, EV_STOP_OP_UNSAT);
      EV_LIVE_CHECK(EV_STOP_RESP_OPCODE, responsible_opcode(s, s.cur(S_STATE), opcode));
    }
  }
  Word2 v{fr_u64(0), fr_u64(0)};
  bool w = false;
  live = need1(s, live, call_context_w(s, live, s.cur(S_RWC), 0, s.cur(S_CALL_ID), ZK_CC_IsSuccess, &v, &w), EV_STOP_CC_UNSAT);
  EV_LIVE_CHECK(EV_STOP_CC_TYPE, !w);
  EV_LIVE_CHECK(EV_STOP_IS_SUCCESS, fr_eq_u64(v.lo, 1));
  const Fr is_root = s.cur(S_IS_ROOT);
  EV_LIVE_CHECK(EV_STOP_ROOT_ENDTX, fr_eq_u64(is_root, fr_eq_u64(s.nxt(S_STATE), ZK_ES_EndTx) ? 1 : 0));
  const bool root = !fr_is_zero(is_root);
  if (live && root) {
    EV_LIVE_CHECK(EV_STOP_RWC, fr_eq(s.nxt(S_RWC), fr_add_u64(s.cur(S_RWC), 1)));
    EV_LIVE_CHECK(EV_STOP_CALL_ID, fr_eq(s.nxt(S_CALL_ID), s.cur(S_CALL_ID)));
  }
  restore_context(s, live && !root, 1, fr_u64(0), fr_u64(0), s.cur(S_GAS), true);
}

// ---- MEMORY: MLOAD / MSTORE / MSTORE8 (execution/memory.py:7-44) -----------------------------
// NB the byte values are NOT constrained by the reference: `instruction.is_equal(memory_lookup(..),
// byte)` only computes a flag (memory.py:26,31-36); each of the 1 / 32 memory rows must exist, be
// unique and hold a value (not a Word).
ZK_HD_NOINLINE void gadget_memory(const StepCtx& s, bool live) {
  Fr opcode = fr_u64(0);
  live = opcode_lookup_ni(s, live, &opcode);
  const Fr rwc = s.cur(S_RWC), call_id = s.cur(S_CALL_ID), sp = s.cur(S_SP);
  const Word2 zero{fr_u64(0), fr_u64(0)};
  Word2 addr_w = zero, val_w = zero;
  live = need1(s, live, rw_lookup_ni(s, live, rwc, 0, ZK_TARGET_Stack, call_id, sp, &addr_w), EV_MEM_ADDR_UNSAT);
  EV_LIVE_CHECK(EV_MEM_ADDR_BYTES, word_in_domain(addr_w));
  EV_LIVE_CHECK(EV_MEM_ADDR_RANGE, (addr_w.hi.l[0] >> 32) == 0 && addr_w.hi.l[1] == 0);  // bytes 20..31 zero
  Fr address = addr_w.lo;
  address.l[2] = addr_w.hi.l[0];  // lo + 2^128 * hi < 2^160
  const bool is_mload = fr_eq_u64(opcode, 0x51), is_mstore8 = fr_eq_u64(opcode, 0x53);
  const bool is_store = !is_mload;
  // value: stack_push() at the popped slot for MLOAD, a second stack_pop() otherwise (memory.py:17)
  live = need1(s, live,
               rw_lookup_ni(s, live, fr_add_u64(rwc, 1), is_mload ? 1 : 0, ZK_TARGET_Stack, call_id,
                         is_mload ? sp : fr_add_u64(sp, 1), &val_w),
               EV_MEM_VAL_UNSAT);
  EV_LIVE_CHECK(EV_MEM_VAL_BYTES, word_in_domain(val_w));
  // memory_expansion(offset = curr.memory_word_size, length = address + 1 + 31 * (1 - is_mstore8)),
  // instruction.py:1138-1155: (length + offset + 31) // 32 must fit 4 bytes, then max() with the
  // current size (both < 2^32)
  const Fr cur_mem = s.cur(S_MEM);
  const Fr num = fr_add_u64(fr_add(fr_add_u64(address, is_mstore8 ? 1 : 32), cur_mem), 31);
  EV_LIVE_CHECK(EV_MEM_MEMSIZE_RANGE, fr_fits64(num) && (num.l[0] >> 37) == 0);
  EV_LIVE_CHECK(EV_MEM_MAX_RANGE, fr_fits64(cur_mem) && (cur_mem.l[0] >> 32) == 0);
  const u64 mem_size = num.l[0] >> 5;
  const u64 nxt = cur_mem.l[0] < mem_size ? mem_size : cur_mem.l[0];
  const int n_bytes = is_mstore8 ? 1 : 32;
  for (int k = 0; k < 32; k++) {  // every lane runs 32 rounds (warp-synchronous lookups)
    const bool go = live && k < n_bytes;
    Fr key[5] = {fr_add_u64(rwc, 2 + k), fr_u64(is_store ? 1 : 0), fr_u64(ZK_TARGET_Memory), call_id,
                 fr_add_u64(address, k)};
    u32 r = 0;
    const int m = lookup_sync<5>(s.t.rw, key, &r, s.mask, go);
    if (go) {
      live = need1(s, live, m, EV_MEM_BYTE_UNSAT);
      EV_LIVE_CHECK(EV_MEM_BYTE_TYPE, !(s.t.rw.tab.flags && (s.t.rw.tab.flags[r] & 1)));
    }
  }
  if (!live) return;
  const Fr gas = fr_u64(memory_gas_cost(nxt) - memory_gas_cost(cur_mem.l[0]));
  same_context_x_ni(s, opcode, fr_u64(is_mstore8 ? 3 : 34), fr_u64(1), fr_u64(is_store ? 2 : 0), true, fr_u64(nxt), gas);
}

// ---- simple same-context gadgets: msize.py, gas.py, iszero.py, comparator.py, jump.py, jumpi.py ----
ZK_HD bool word_is(const Word2& w, const Fr& lo) { return fr_eq(w.lo, lo) && fr_is_zero(w.hi); }
// one stack_push / stack_pop lookup at rw_counter + k
ZK_HD_NOINLINE int stack_at(const StepCtx& s, bool live, u64 k, u64 rw, const Fr& sp, Word2* out) {
  return rw_lookup_ni(s, live, fr_add_u64(s.cur(S_RWC), k), rw, ZK_TARGET_Stack, s.cur(S_CALL_ID), sp, out);
}
ZK_HD_NOINLINE void gadget_msize(const StepCtx& s, bool live) {
  Fr opcode = fr_u64(0);
  live = opcode_lookup_ni(s, live, &opcode);
  const Fr v = fr_montmul(s.cur(S_MEM), fr_to_mont(fr_u64(32)));  // memory_word_size * N_BYTES_WORD over the field
  EV_LIVE_CHECK(EV_MSZ_WORD, fr_fits128(v));
  Word2 w{fr_u64(0), fr_u64(0)};
  live = need1(s, live, stack_at(s, live, 0, 1, fr_sub_u64(s.cur(S_SP), 1), &w), EV_MSZ_PUSH_UNSAT);
  EV_LIVE_CHECK(EV_MSZ_EQ, word_is(w, v));
  if (!live) return;
  same_context_ni(s, opcode, 1, fr_u64(1), fr_sub(fr_u64(0), fr_u64(1)));
}
ZK_HD_NOINLINE void gadget_gas(const StepCtx& s, bool live) {
  Fr opcode = fr_u64(0);
  live = opcode_lookup_ni(s, live, &opcode);
  EV_LIVE_CHECK(EV_GAS_OPCODE, fr_eq_u64(opcode, 0x5a));
  const Fr v = fr_sub_u64(s.cur(S_GAS), 2);  // Opcode.GAS.constant_gas_cost() == 2
  EV_LIVE_CHECK(EV_GAS_WORD, fr_fits128(v));
  Word2 w{fr_u64(0), fr_u64(0)};
  live = need1(s, live, stack_at(s, live, 0, 1, fr_sub_u64(s.cur(S_SP), 1), &w), EV_GAS_PUSH_UNSAT);
  EV_LIVE_CHECK(EV_GAS_EQ, word_is(w, v));
  if (!live) return;
  same_context_ni(s, opcode, 1, fr_u64(1), fr_sub(fr_u64(0), fr_u64(1)));
}
ZK_HD_NOINLINE void gadget_iszero(const StepCtx& s, bool live) {
  Fr opcode = fr_u64(0);
  live = opcode_lookup_ni(s, live, &opcode);
  Word2 v{fr_u64(0), fr_u64(0)}, w{fr_u64(0), fr_u64(0)};
  live = need1(s, live, stack_at(s, live, 0, 0, s.cur(S_SP), &v), EV_ISZ_POP_UNSAT);
  live = need1(s, live, stack_at(s, live, 1, 1, s.cur(S_SP), &w), EV_ISZ_PUSH_UNSAT);
  EV_LIVE_CHECK(EV_ISZ_EQ, word_is(w, fr_u64(fr_is_zero(fr_add(v.lo, v.hi)) ? 1 : 0)));  // is_zero_word: field sum
  if (!live) return;
  same_context_ni(s, opcode, 2, fr_u64(1), fr_u64(0));
}
ZK_HD_NOINLINE void gadget_cmp(const StepCtx& s, bool live) {
  Fr opcode = fr_u64(0);
  live = opcode_lookup_ni(s, live, &opcode);
  const bool is_eq = fr_eq_u64(opcode, 0x14), is_gt = fr_eq_u64(opcode, 0x11);
  const Fr sp = s.cur(S_SP), sp1 = fr_add_u64(sp, 1);
  const Word2 zero{fr_u64(0), fr_u64(0)};
  Word2 a = zero, b = zero, c = zero;
  live = need1(s, live, stack_at(s, live, 0, 0, sp, &a), EV_CMP_A_UNSAT);
  live = need1(s, live, stack_at(s, live, 1, 0, sp1, &b), EV_CMP_B_UNSAT);
  live = need1(s, live, stack_at(s, live, 2, 1, sp1, &c), EV_CMP_C_UNSAT);
  const Word2 aa = is_gt ? b : a, bb = is_gt ? a : b;  // comparator.py:18 swap for GT
  EV_LIVE_CHECK(EV_CMP_RANGE_LO, fr_fits128(aa.lo) && fr_fits128(bb.lo));
  EV_LIVE_CHECK(EV_CMP_RANGE_HI, fr_fits128(aa.hi) && fr_fits128(bb.hi));
  const bool lt_lo = fr_lt(aa.lo, bb.lo), eq_lo = fr_eq(aa.lo, bb.lo), lt_hi = fr_lt(aa.hi, bb.hi), eq_hi = fr_eq(aa.hi, bb.hi);
  const bool lt = lt_hi || (eq_hi && lt_lo), eq = eq_lo && eq_hi;
  EV_LIVE_CHECK(EV_CMP_EQ, word_is(c, fr_u64((is_eq ? eq : lt) ? 1 : 0)));
  if (!live) return;
  same_context_ni(s, opcode, 3, fr_u64(1), fr_u64(1));
}
ZK_HD_NOINLINE void gadget_jump(const StepCtx& s, bool live) {
  Fr opcode = fr_u64(0);
  live = opcode_lookup_ni(s, live, &opcode);
  EV_LIVE_CHECK(EV_JMP_OPCODE, fr_eq_u64(opcode, 0x56));
  Word2 dest{fr_u64(0), fr_u64(0)};
  live = need1(s, live, stack_at(s, live, 0, 0, s.cur(S_SP), &dest), EV_JMP_DEST_UNSAT);
  EV_LIVE_CHECK(EV_JMP_DEST_HI, fr_is_zero(dest.hi));
  Fr at = fr_u64(0);  // opcode_lookup_at(dest, True), instruction.py:789-790
  live = need1(s, live, bytecode_lookup_ni(s, live, s.cur(S_HASH_LO), s.cur(S_HASH_HI), 2, dest.lo, 1, &at), EV_JMP_AT_UNSAT);
  EV_LIVE_CHECK(EV_JMP_NOT_JUMPDEST, fr_eq_u64(at, 0x5b));
  if (!live) return;
  // program_counter = Transition.to(dest): next.pc == dest, i.e. the delta dest - pc over the field
  same_context_ni(s, opcode, 1, fr_sub(dest.lo, s.cur(S_PC)), fr_u64(1));
}
ZK_HD_NOINLINE void gadget_jumpi(const StepCtx& s, bool live) {
  Fr opcode = fr_u64(0);
  live = opcode_lookup_ni(s, live, &opcode);
  EV_LIVE_CHECK(EV_JMPI_OPCODE, fr_eq_u64(opcode, 0x57));
  Word2 dest{fr_u64(0), fr_u64(0)}, cond{fr_u64(0), fr_u64(0)};
  live = need1(s, live, stack_at(s, live, 0, 0, s.cur(S_SP), &dest), EV_JMPI_DEST_UNSAT);
  EV_LIVE_CHECK(EV_JMPI_DEST_HI, fr_is_zero(dest.hi));
  live = need1(s, live, stack_at(s, live, 1, 0, fr_add_u64(s.cur(S_SP), 1), &cond), EV_JMPI_COND_UNSAT);
  if (!live) return;
  // jumpi.py:20 `if instruction.is_zero_word(cond):` tests the truthiness of an FQ OBJECT (py_ecc's FQ
  // defines neither __bool__ nor __len__), which is always true: the reference takes the fall-through
  // branch (pc + 1) whatever cond is and never looks at the destination.  Reproduced as written.
  same_context_ni(s, opcode, 2, fr_u64(1), fr_u64(2));
}

// caller.py / callvalue.py / calldatasize.py / address.py / returndatasize.py: constrain the opcode,
// read one call-context field (as a Word, or as a value wrapped by Word.from_lo), push it
ZK_HD_NOINLINE void gadget_cc_push(const StepCtx& s, bool live, u64 op, u64 field, bool as_word) {
  Fr opcode = fr_u64(0);
  live = opcode_lookup_ni(s, live, &opcode);
  EV_LIVE_CHECK(EV_CCP_OPCODE, fr_eq_u64(opcode, op));
  Word2 v{fr_u64(0), fr_u64(0)}, w{fr_u64(0), fr_u64(0)};
  bool is_word = false;
  live = need1(s, live, call_context_w(s, live, s.cur(S_RWC), 0, s.cur(S_CALL_ID), field, &v, &is_word), EV_CCP_CC_UNSAT);
  if (!as_word) {
    EV_LIVE_CHECK(EV_CCP_CC_TYPE, !is_word);
    EV_LIVE_CHECK(EV_CCP_WORD, fr_fits128(v.lo));
    v.hi = fr_u64(0);
  }
  live = need1(s, live, stack_at(s, live, 1, 1, fr_sub_u64(s.cur(S_SP), 1), &w), EV_CCP_PUSH_UNSAT);
  EV_LIVE_CHECK(EV_CCP_EQ, word_eq(w, v));
  if (!live) return;
  same_context_ni(s, opcode, 2, fr_u64(1), fr_sub(fr_u64(0), fr_u64(1)));
}
ZK_HD_NOINLINE void gadget_codesize(const StepCtx& s, bool live) {
  Fr opcode = fr_u64(0);
  live = opcode_lookup_ni(s, live, &opcode);
  EV_LIVE_CHECK(EV_CSZ_OPCODE, fr_eq_u64(opcode, 0x38));
  Fr len = fr_u64(0);  // bytecode_length(code_hash): the Header row (instruction.py:772-777)
  live = need1(s, live, bytecode_lookup_ni(s, live, s.cur(S_HASH_LO), s.cur(S_HASH_HI), 1, fr_u64(0), 0, &len), EV_CSZ_LEN_UNSAT);
  EV_LIVE_CHECK(EV_CSZ_WORD, fr_fits128(len));
  Word2 w{fr_u64(0), fr_u64(0)};
  live = need1(s, live, stack_at(s, live, 0, 1, fr_sub_u64(s.cur(S_SP), 1), &w), EV_CSZ_PUSH_UNSAT);
  EV_LIVE_CHECK(EV_CSZ_EQ, word_is(w, len));
  if (!live) return;
  same_context_ni(s, opcode, 1, fr_u64(1), fr_sub(fr_u64(0), fr_u64(1)));
}

// ---- BITWISE = AND / OR / XOR (bitwise.py), NOT (not_.py), BYTE (byte.py) ------------------------
ZK_HD u64 word_byte(const Word2& w, int k) {  // k-th little-endian byte of a word in the 128-bit-halves domain
  const Fr& c = k < 16 ? w.lo : w.hi;
  k &= 15;
  return (c.l[k >> 3] >> (8 * (k & 7))) & 0xFF;
}
// 32 fixed-table lookups (tag, a[i], b[i], c[i]); returns false after recording the first failure
ZK_HD_NOINLINE bool fixed_bytes32(const StepCtx& s, bool live, u64 tag, const Word2& a, const Word2& b, const Word2* c, u64 c_const,
                         int id_unsat) {
  for (int k = 0; k < 32; k++) {
    Fr key[4] = {fr_u64(tag), fr_u64(word_byte(a, k)), fr_u64(word_byte(b, k)), fr_u64(c ? word_byte(*c, k) : c_const)};
    u32 r = 0;
    const int m = lookup_sync<4>(s.t.fixed, key, &r, s.mask, live);
    live = need1(s, live, m, id_unsat);
  }
  return live;
}
ZK_HD_NOINLINE void gadget_bitwise(const StepCtx& s, bool live) {
  Fr opcode = fr_u64(0);
  live = opcode_lookup_ni(s, live, &opcode);
  const Fr sp = s.cur(S_SP), sp1 = fr_add_u64(sp, 1);
  const Word2 zero{fr_u64(0), fr_u64(0)};
  Word2 a = zero, b = zero, c = zero;
  live = need1(s, live, stack_at(s, live, 0, 0, sp, &a), EV_BW_A_UNSAT);
  live = need1(s, live, stack_at(s, live, 1, 0, sp1, &b), EV_BW_B_UNSAT);
  live = need1(s, live, stack_at(s, live, 2, 1, sp1, &c), EV_BW_C_UNSAT);
  EV_LIVE_CHECK(EV_BW_BYTES, word_in_domain(a) && word_in_domain(b) && word_in_domain(c));
  // tag = BitwiseAnd + (opcode.n - AND) as a Python int; FixedTableTag(tag) must exist (1..16)
  EV_LIVE_CHECK(EV_BW_TAG, fr_fits64(opcode) && opcode.l[0] >= 0x16 - 9 && opcode.l[0] <= 0x16 + 6);
  const u64 tag = opcode.l[0] + ZK_FIXED_BitwiseAnd - 0x16;
  live = fixed_bytes32(s, live, tag, a, b, &c, 0, EV_BW_FIXED_UNSAT);
  if (!live) return;
  same_context_ni(s, opcode, 3, fr_u64(1), fr_u64(1));
}
ZK_HD_NOINLINE void gadget_not(const StepCtx& s, bool live) {
  Fr opcode = fr_u64(0);
  live = opcode_lookup_ni(s, live, &opcode);
  const Word2 zero{fr_u64(0), fr_u64(0)};
  Word2 a = zero, b = zero;
  live = need1(s, live, stack_at(s, live, 0, 0, s.cur(S_SP), &a), EV_NOT_A_UNSAT);
  EV_LIVE_CHECK(EV_NOT_A_BYTES, word_in_domain(a));
  live = need1(s, live, stack_at(s, live, 1, 1, s.cur(S_SP), &b), EV_NOT_B_UNSAT);
  EV_LIVE_CHECK(EV_NOT_B_BYTES, word_in_domain(b));
  live = fixed_bytes32(s, live, ZK_FIXED_BitwiseXor, a, b, nullptr, 255, EV_NOT_FIXED_UNSAT);
  if (!live) return;
  same_context_ni(s, opcode, 2, fr_u64(1), fr_u64(0));
}
ZK_HD_NOINLINE void gadget_byte(const StepCtx& s, bool live) {
  Fr opcode = fr_u64(0);
  live = opcode_lookup_ni(s, live, &opcode);
  const Fr sp = s.cur(S_SP), sp1 = fr_add_u64(sp, 1);
  const Word2 zero{fr_u64(0), fr_u64(0)};
  Word2 a = zero, b = zero, c = zero;
  live = need1(s, live, stack_at(s, live, 0, 0, sp, &a), EV_BYTE_A_UNSAT);
  live = need1(s, live, stack_at(s, live, 1, 0, sp1, &b), EV_BYTE_B_UNSAT);
  live = need1(s, live, stack_at(s, live, 2, 1, sp1, &c), EV_BYTE_C_UNSAT);
  EV_LIVE_CHECK(EV_BYTE_BYTES, word_in_domain(a) && word_in_domain(b));
  if (!live) return;
  // byte.py:16-29: index bytes 1..31 all zero and index[0] < 32 select value byte 31 - index[0], else 0
  const bool msb_zero = (a.lo.l[0] >> 8) == 0 && a.lo.l[1] == 0 && a.hi.l[0] == 0 && a.hi.l[1] == 0;
  const u64 idx0 = a.lo.l[0] & 0xFF;
  const u64 sel = (msb_zero && idx0 < 32) ? word_byte(b, 31 - (int)idx0) : 0;
  EV_CHECK(EV_BYTE_EQ, word_is(c, fr_u64(sel)));
  same_context_ni(s, opcode, 3, fr_u64(1), fr_u64(1));
}

// ---- SCMP = SLT / SGT (slt_sgt.py), SIGNEXTEND (signextend.py) -----------------------------------
ZK_HD_NOINLINE void gadget_scmp(const StepCtx& s, bool live) {
  Fr opcode = fr_u64(0);
  live = opcode_lookup_ni(s, live, &opcode);
  const bool is_sgt = fr_eq_u64(opcode, 0x13);
  const Fr sp = s.cur(S_SP), sp1 = fr_add_u64(sp, 1);
  const Word2 zero{fr_u64(0), fr_u64(0)};
  Word2 a = zero, b = zero, c = zero;
  live = need1(s, live, stack_at(s, live, 0, 0, sp, &a), EV_SCMP_A_UNSAT);
  live = need1(s, live, stack_at(s, live, 1, 0, sp1, &b), EV_SCMP_B_UNSAT);
  live = need1(s, live, stack_at(s, live, 2, 1, sp1, &c), EV_SCMP_C_UNSAT);
  if (!live) return;
  const Word2 aa = is_sgt ? b : a, bb = is_sgt ? a : b;  // slt_sgt.py:17-18 swap for SGT
  EV_CHECK(EV_SCMP_BYTES, word_in_domain(aa) && word_in_domain(bb) && word_in_domain(c));
  EV_CHECK(EV_SCMP_C_MSB, word_byte(c, 31) == 0);
  const bool lt_lo = fr_lt(aa.lo, bb.lo), lt_hi = fr_lt(aa.hi, bb.hi), eq_hi = fr_eq(aa.hi, bb.hi);
  const bool a_lt_b = lt_hi || (eq_hi && lt_lo);
  const bool a_neg = word_byte(aa, 31) >= 128, b_neg = word_byte(bb, 31) >= 128;
  const bool expect = (a_neg && !b_neg) ? true : ((b_neg && !a_neg) ? false : a_lt_b);
  EV_CHECK(EV_SCMP_EQ, word_is(c, fr_u64(expect ? 1 : 0)));  // cc = low 31 bytes of c; byte 31 is zero here
  same_context_ni(s, opcode, 3, fr_u64(1), fr_u64(1));
}
// signextend.py: the byte-by-byte `is_equal` calls constrain nothing; what remains is the
// sign_byte_lookup of the selected byte (signextend.py:44) — note that sign_byte ignores
// is_msb_sum_zero while selected_byte does not (reproduced)
ZK_HD_NOINLINE void gadget_signextend(const StepCtx& s, bool live) {
  Fr opcode = fr_u64(0);
  live = opcode_lookup_ni(s, live, &opcode);
  const Fr sp = s.cur(S_SP), sp1 = fr_add_u64(sp, 1);
  const Word2 zero{fr_u64(0), fr_u64(0)};
  Word2 index = zero, value = zero, result = zero;
  live = need1(s, live, stack_at(s, live, 0, 0, sp, &index), EV_SEXT_IDX_UNSAT);
  live = need1(s, live, stack_at(s, live, 1, 0, sp1, &value), EV_SEXT_VAL_UNSAT);
  live = need1(s, live, stack_at(s, live, 2, 1, sp1, &result), EV_SEXT_RES_UNSAT);
  EV_LIVE_CHECK(EV_SEXT_BYTES, word_in_domain(index) && word_in_domain(value) && word_in_domain(result));
  const bool msb_zero = (index.lo.l[0] >> 8) == 0 && index.lo.l[1] == 0 && index.hi.l[0] == 0 && index.hi.l[1] == 0;
  const u64 idx0 = index.lo.l[0] & 0xFF;
  const u64 vbyte = idx0 < 31 ? word_byte(value, (int)idx0) : 0;
  const u64 sign_byte = (vbyte >> 7) * 0xFF, selected = msb_zero ? vbyte : 0;
  {
    Fr key[4] = {fr_u64(ZK_FIXED_SignByte), fr_u64(selected), fr_u64(sign_byte), fr_u64(0)};
    u32 r = 0;
    const int m = lookup_sync<4>(s.t.fixed, key, &r, s.mask, live);
    live = need1(s, live, m, EV_SEXT_SIGN_UNSAT);
  }
  if (!live) return;
  same_context_ni(s, opcode, 3, fr_u64(1), fr_u64(1));
}

// ---- BlockCtx (block_ctx.py: COINBASE / TIMESTAMP / NUMBER / PREVRANDAO / GASLIMIT / CHAINID / BASEFEE),
// ORIGIN (origin.py), GASPRICE (gasprice.py): a block-table / tx-table word pushed on the stack -----
ZK_HD_NOINLINE void gadget_blockctx(const StepCtx& s, bool live) {
  Fr opcode = fr_u64(0);
  live = opcode_lookup_ni(s, live, &opcode);
  u64 tag = 0;  // BlockContextFieldTag of the opcode (block_ctx.py:10-24); none: `op` stays unbound
  if (fr_fits64(opcode)) switch (opcode.l[0]) {
      case 0x41: tag = 1; break;  // COINBASE -> Coinbase
      case 0x42: tag = 4; break;  // TIMESTAMP
      case 0x43: tag = 3; break;  // NUMBER
      case 0x45: tag = 2; break;  // GASLIMIT
      case 0x44: tag = 5; break;  // PREVRANDAO
      case 0x48: tag = 6; break;  // BASEFEE
      case 0x46: tag = 7; break;  // CHAINID
      default: break;
    }
  EV_LIVE_CHECK(EV_BLK_OPCODE, tag != 0);
  Word2 ctx{fr_u64(0), fr_u64(0)}, w{fr_u64(0), fr_u64(0)};
  {
    Fr key[2] = {fr_u64(tag), fr_u64(0)};
    u32 r = 0;
    const int m = lookup_sync<2>(s.t.block, key, &r, s.mask, live);
    live = need1(s, live, m, EV_BLK_CTX_UNSAT);
    if (live) {
      ctx.lo = table_cell(s.t.block.tab, 2, r);
      ctx.hi = table_cell(s.t.block.tab, 3, r);
    }
  }
  live = need1(s, live, stack_at(s, live, 0, 1, fr_sub_u64(s.cur(S_SP), 1), &w), EV_BLK_PUSH_UNSAT);
  EV_LIVE_CHECK(EV_BLK_EQ, word_eq(w, ctx));
  if (!live) return;
  same_context_ni(s, opcode, 1, fr_u64(1), fr_sub(fr_u64(0), fr_u64(1)));
}
ZK_HD_NOINLINE void gadget_txctx(const StepCtx& s, bool live, u64 op, u64 field) {
  // the call-context lookup comes BEFORE the opcode lookup here (origin.py:8-9)
  Word2 v{fr_u64(0), fr_u64(0)}, ctx{fr_u64(0), fr_u64(0)}, w{fr_u64(0), fr_u64(0)};
  bool is_word = false;
  live = need1(s, live, call_context_w(s, live, s.cur(S_RWC), 0, s.cur(S_CALL_ID), ZK_CC_TxId, &v, &is_word), EV_TXC_TXID_UNSAT);
  EV_LIVE_CHECK(EV_TXC_TXID_TYPE, !is_word);
  Fr opcode = fr_u64(0);
  live = opcode_lookup_ni(s, live, &opcode);
  EV_LIVE_CHECK(EV_TXC_OPCODE, fr_eq_u64(opcode, op));
  {
    Fr key[3] = {v.lo, fr_u64(field), fr_u64(0)};
    u32 r = 0;
    const int m = lookup_sync<3>(s.t.tx, key, &r, s.mask, live);
    live = need1(s, live, m, EV_TXC_TX_UNSAT);
    if (live) {
      ctx.lo = table_cell(s.t.tx.tab, 3, r);
      ctx.hi = table_cell(s.t.tx.tab, 4, r);
    }
  }
  live = need1(s, live, stack_at(s, live, 1, 1, fr_sub_u64(s.cur(S_SP), 1), &w), EV_TXC_PUSH_UNSAT);
  EV_LIVE_CHECK(EV_TXC_EQ, word_eq(w, ctx));
  if (!live) return;
  same_context_ni(s, opcode, 2, fr_u64(1), fr_sub(fr_u64(0), fr_u64(1)));
}

// ---- SHL_SHR (shl_shr.py): push == pop2 << pop1 / pop2 >> pop1 through a division witness --------
// unsigned 640-bit integers: Word.int_value() of arbitrary cells is < 2^382 and the SHR remainder
// witness is dividend - quotient * 2^shift (shift < 256), all as Python ints in the reference
struct U640 {
  u64 l[10];
};
ZK_HD U640 word_int(const Word2& w) {  // lo + hi * 2^128 as an integer
  U640 r;
  for (int k = 0; k < 10; k++) r.l[k] = 0;
  u64 c = 0;
  r.l[0] = w.lo.l[0];
  r.l[1] = w.lo.l[1];
  r.l[2] = adc64(w.lo.l[2], w.hi.l[0], c);
  r.l[3] = adc64(w.lo.l[3], w.hi.l[1], c);
  r.l[4] = adc64(w.hi.l[2], 0, c);
  r.l[5] = adc64(w.hi.l[3], 0, c);
  r.l[6] = c;
  return r;
}
ZK_HD U640 u640_shl(const U640& a, unsigned sh) {  // sh < 256
  U640 r;
  const int ws = (int)(sh >> 6);
  const unsigned bs = sh & 63;
  for (int k = 9; k >= 0; k--) {
    u64 v = 0;
    if (k >= ws) {
      v = a.l[k - ws] << bs;
      if (bs && k - ws - 1 >= 0) v |= a.l[k - ws - 1] >> (64 - bs);
    }
    r.l[k] = v;
  }
  return r;
}
ZK_HD int u640_cmp(const U640& a, const U640& b) {
  for (int k = 9; k >= 0; k--) {
    if (a.l[k] < b.l[k]) return -1;
    if (a.l[k] > b.l[k]) return 1;
  }
  return 0;
}
ZK_HD U640 u640_sub(const U640& a, const U640& b) {
  U640 r;
  u64 br = 0;
  for (int k = 0; k < 10; k++) r.l[k] = sbb64(a.l[k], b.l[k], br);
  return r;
}
ZK_HD_NOINLINE void gadget_shl_shr(const StepCtx& s, bool live) {
  Fr opcode = fr_u64(0);
  live = opcode_lookup_ni(s, live, &opcode);
  const Fr sp = s.cur(S_SP), sp1 = fr_add_u64(sp, 1), one = fr_u64(1);
  const Word2 zero{fr_u64(0), fr_u64(0)};
  Word2 pop1 = zero, pop2 = zero, push = zero;
  live = need1(s, live, stack_at(s, live, 0, 0, sp, &pop1), EV_SH_P1_UNSAT);
  live = need1(s, live, stack_at(s, live, 1, 0, sp1, &pop2), EV_SH_P2_UNSAT);
  live = need1(s, live, stack_at(s, live, 2, 1, sp1, &push), EV_SH_PUSH_UNSAT);
  // gen_witness, shl_shr.py:103-129
  const Fr is_shl = fr_sub(fr_u64(0x1c), opcode);  // Opcode.SHR - opcode over the field
  EV_LIVE_CHECK(EV_SH_BYTES, word_in_domain(pop1));
  const unsigned shf0 = (unsigned)word_byte(pop1, 0);
  const bool shf_lt256 = (pop1.lo.l[0] >> 8) == 0 && pop1.lo.l[1] == 0 && pop1.hi.l[0] == 0 && pop1.hi.l[1] == 0;
  Word2 divisor = zero;  // Word(1 << shf0) if the shift is < 256 else Word(0)
  if (shf_lt256) {
    const u64 bit = 1ull << (shf0 & 63);
    if (shf0 < 64) divisor.lo.l[0] = bit;
    else if (shf0 < 128) divisor.lo.l[1] = bit;
    else if (shf0 < 192) divisor.hi.l[0] = bit;
    else divisor.hi.l[1] = bit;
  }
  Word2 dividend, quotient, remainder = zero;
  if (fr_eq_u64(is_shl, 1)) {
    dividend = push;
    quotient = pop2;
  } else {
    dividend = pop2;
    quotient = push;
    if (live) {
      // remainder = Word(dividend.int_value() - quotient.int_value() * divisor.int_value()) as Python ints
      const U640 D = word_int(dividend);
      U640 QS;
      for (int k = 0; k < 10; k++) QS.l[k] = 0;
      if (shf_lt256) QS = u640_shl(word_int(quotient), shf0);
      EV_LIVE_CHECK(EV_SH_REM_NEG, u640_cmp(D, QS) >= 0);  // Word(negative).to_bytes -> OverflowError
      if (live) {
        const U640 R = u640_sub(D, QS);
        EV_LIVE_CHECK(EV_SH_REM_WORD, (R.l[4] | R.l[5] | R.l[6] | R.l[7] | R.l[8] | R.l[9]) == 0);  // assert < 256**32
        remainder.lo = fr_u128(R.l[0], R.l[1]);
        remainder.hi = fr_u128(R.l[2], R.l[3]);
      }
    }
  }
  if (!live) {  // the pow2 lookup below is warp-synchronous: take part in it, inactive
    Fr key[4] = {fr_u64(0), fr_u64(0), fr_u64(0), fr_u64(0)};
    u32 r = 0;
    lookup_sync<4>(s.t.fixed, key, &r, s.mask, false);
    return;
  }
  // check_witness, shl_shr.py:37-91
  const Fr is_shr = fr_sub(one, is_shl);
  const bool dz = fr_is_zero(fr_add(divisor.lo, divisor.hi));
  Word2 t1, t2, sum;
  bool ok = word_select(quotient, is_shl, &t1) && word_select(dividend, is_shr, &t2);  // :59-62
  sum.lo = fr_add(t1.lo, t2.lo);
  sum.hi = fr_add(t1.hi, t2.hi);
  int fail_id = -1;
  if (!(ok && word_in_domain(sum))) fail_id = EV_SH_SELECT;
  else if (!word_eq(pop2, sum)) fail_id = EV_SH_POP2;
  if (fail_id < 0) {  // :63-65
    ok = word_select(dividend, is_shl, &t1) && word_select(quotient, dz ? fr_u64(0) : is_shr, &t2);
    sum.lo = fr_add(t1.lo, t2.lo);
    sum.hi = fr_add(t1.hi, t2.hi);
    if (!(ok && word_in_domain(sum))) fail_id = EV_SH_SELECT;
    else if (!word_eq(push, sum)) fail_id = EV_SH_PUSH_EQ;
  }
  // :66-76 hold by construction of shf0 / divisor (the shift is in the bytes domain here)
  if (fail_id < 0) {  // :77-79 compare_word(remainder, divisor), both in the halves domain
    const bool lt = fr_lt(remainder.hi, divisor.hi) || (fr_eq(remainder.hi, divisor.hi) && fr_lt(remainder.lo, divisor.lo));
    if (!(dz || lt)) fail_id = EV_SH_REM_LT;
  }
  if (fail_id < 0 && !fr_is_zero(is_shl) && !(fr_is_zero(remainder.lo) && fr_is_zero(remainder.hi))) fail_id = EV_SH_SHL_REM0;
  if (fail_id < 0 && !word_in_domain(quotient)) fail_id = EV_SH_TO64;  // :86 mul_add_words(quotient, divisor, remainder, dividend)
  if (fail_id < 0) {
    Fr carry_lo, carry_hi, overflow;
    mul_add_carries(quotient, divisor, remainder, dividend, &carry_lo, &carry_hi, &overflow);
    if (!fits_9_bytes(carry_lo)) fail_id = EV_SH_CARRY_LO;
    else if (!fits_9_bytes(carry_hi)) fail_id = EV_SH_CARRY_HI;
    else if (!(fr_is_zero(is_shr) || fr_is_zero(overflow))) fail_id = EV_SH_OVERFLOW;
  }
  if (fail_id >= 0) {
    step_fail(s, fail_id);
    live = false;
  }
  {  // :90-91 pow2_lookup(shf0, divisor_lo, divisor_hi) when the divisor is not zero
    const bool go = live && !dz;
    Fr key[4] = {fr_u64(ZK_FIXED_Pow2), fr_u64(shf0), divisor.lo, divisor.hi};
    u32 r = 0;
    const int m = lookup_sync<4>(s.t.fixed, key, &r, s.mask, go);
    if (go) live = need1(s, live, m, EV_SH_POW2_UNSAT);
  }
  if (!live) return;
  same_context_ni(s, opcode, 3, one, one);
}

}  // namespace zk
#include "evm_tx.cuh"
#include "evm_err.cuh"
#include "evm_arith.cuh"
#include "evm_storage.cuh"
#include "evm_log.cuh"
#include "evm_exp.cuh"
#include "evm_return.cuh"
#include "evm_call.cuh"
#include "evm_create.cuh"
namespace zk {

// ---- gate-program groups --------------------------------------------------------------------
// One kernel per GROUP of gate programs with similar register needs; inside a group kernel every
// execution state has its own bucket of steps, so warps run one gate program (k_evm_classify /
// k_evm_scatter sort the steps by state).  The host launches a group only when one of its buckets is
// non-empty (zk_check_async reads the histogram back).
enum { KG_ADD, KG_MUL, KG_PUSH, KG_POP, KG_SIMPLE, KG_BYTES32, KG_COPY, KG_WIDE, KG_TX, KG_ARITH, KG_COUNT };
__host__ __device__ constexpr int es_group(int st) {
  switch (st) {
    case ZK_ES_ADD: return KG_ADD;
    case ZK_ES_MUL: case ZK_BK_DIV: case ZK_BK_MOD: return KG_MUL;
    case ZK_ES_PUSH: return KG_PUSH;
    case ZK_ES_POP: return KG_POP;
    case ZK_ES_MSIZE: case ZK_ES_GAS: case ZK_ES_ISZERO: case ZK_ES_CMP: case ZK_ES_JUMP: case ZK_ES_JUMPI:
    case ZK_ES_CALLER: case ZK_ES_CALLVALUE: case ZK_ES_CALLDATASIZE: case ZK_ES_ADDRESS: case ZK_ES_RETURNDATASIZE:
    case ZK_ES_CODESIZE: case ZK_ES_BYTE: case ZK_ES_SCMP: case ZK_ES_SIGNEXTEND: case ZK_ES_BlockCtx:
    case ZK_ES_ORIGIN: case ZK_ES_GASPRICE: return KG_SIMPLE;
    case ZK_ES_BITWISE: case ZK_ES_NOT: case ZK_ES_MEMORY: return KG_BYTES32;
    case ZK_ES_SHA3: case ZK_ES_CALLDATACOPY: return KG_COPY;
    case ZK_ES_SHL_SHR: return KG_WIDE;
    case ZK_ES_ADDMOD: case ZK_ES_MULMOD: case ZK_ES_SDIV_SMOD: case ZK_ES_SAR: case ZK_ES_EXP: return KG_ARITH;
    case ZK_ES_STOP: case ZK_ES_BeginTx: case ZK_ES_EndTx: case ZK_ES_EndBlock: case ZK_ES_ErrorStack:
    case ZK_ES_ErrorInvalidOpcode: case ZK_ES_ErrorOutOfGasConstant: case ZK_ES_ErrorInvalidJump: case ZK_ES_SELFBALANCE:
    case ZK_ES_ErrorOutOfGasSHA3: case ZK_ES_ErrorOutOfGasStaticMemoryExpansion: case ZK_ES_ErrorOutOfGasDynamicMemoryExpansion:
    case ZK_ES_ErrorOutOfGasLOG: case ZK_ES_ErrorOutOfGasEXP: case ZK_ES_ErrorReturnDataOutOfBound:
    case ZK_ES_BALANCE: case ZK_ES_EXTCODEHASH: case ZK_ES_EXTCODESIZE: case ZK_ES_ErrorOutOfGasAccountAccess:
    case ZK_ES_CODECOPY: case ZK_ES_RETURNDATACOPY: case ZK_ES_EXTCODECOPY: case ZK_ES_ErrorOutOfGasMemoryCopy:
    case ZK_ES_SLOAD: case ZK_ES_SSTORE: case ZK_ES_CALLDATALOAD: case ZK_ES_LOG: case ZK_ES_ErrorWriteProtection: case ZK_ES_BLOCKHASH:
    case ZK_ES_ErrorMaxCodeSizeExceeded: case ZK_ES_ErrorOutOfGasCodeStore: case ZK_ES_ErrorInvalidCreationCode:
    case ZK_ES_RETURN: case ZK_ES_ErrorOutOfGasCall: case ZK_ES_CALL_OP: case ZK_ES_CREATE: case ZK_ES_CREATE2:
    case ZK_ES_ErrorOutOfGasSloadSstore: case ZK_ES_ErrorOutOfGasCREATE: case ZK_ES_ErrorOutOfGasPrecompile:
    case ZK_ES_ErrorGasUintOverflow:
      return KG_TX;
    default: return -1;
  }
}
// the rare gate programs of one group (st = execution state; other states: nothing)
// `flags`: ZK_FLAG_EVM_* of the check (BeginTx / EndBlock look at the first / last step rules, main.py:47-56)
template <int G>
ZK_HD void run_group(const StepCtx& s, int st, u32 flags) {
  if constexpr (G == KG_SIMPLE) {
    switch (st) {
      case ZK_ES_MSIZE: gadget_msize(s, true); break;
      case ZK_ES_GAS: gadget_gas(s, true); break;
      case ZK_ES_ISZERO: gadget_iszero(s, true); break;
      case ZK_ES_CMP: gadget_cmp(s, true); break;
      case ZK_ES_JUMP: gadget_jump(s, true); break;
      case ZK_ES_JUMPI: gadget_jumpi(s, true); break;
      case ZK_ES_CALLER: gadget_cc_push(s, true, 0x33, ZK_CC_CallerAddress, true); break;
      case ZK_ES_CALLVALUE: gadget_cc_push(s, true, 0x34, ZK_CC_Value, true); break;
      case ZK_ES_CALLDATASIZE: gadget_cc_push(s, true, 0x36, ZK_CC_CallDataLength, false); break;
      case ZK_ES_ADDRESS: gadget_cc_push(s, true, 0x30, ZK_CC_CalleeAddress, true); break;
      case ZK_ES_RETURNDATASIZE: gadget_cc_push(s, true, 0x3d, ZK_CC_LastCalleeReturnDataLength, false); break;
      case ZK_ES_CODESIZE: gadget_codesize(s, true); break;
      case ZK_ES_BYTE: gadget_byte(s, true); break;
      case ZK_ES_SCMP: gadget_scmp(s, true); break;
      case ZK_ES_SIGNEXTEND: gadget_signextend(s, true); break;
      case ZK_ES_BlockCtx: gadget_blockctx(s, true); break;
      case ZK_ES_ORIGIN: gadget_txctx(s, true, 0x32, ZK_TX_CallerAddress); break;
      case ZK_ES_GASPRICE: gadget_txctx(s, true, 0x3a, ZK_TX_GasPrice); break;
      default: break;
    }
  } else if constexpr (G == KG_BYTES32) {
    switch (st) {
      case ZK_ES_BITWISE: gadget_bitwise(s, true); break;
      case ZK_ES_NOT: gadget_not(s, true); break;
      case ZK_ES_MEMORY: gadget_memory(s, true); break;
      default: break;
    }
  } else if constexpr (G == KG_COPY) {
    switch (st) {
      case ZK_ES_SHA3: gadget_sha3(s, true); break;
      case ZK_ES_CALLDATACOPY: gadget_calldatacopy(s, true); break;
      default: break;
    }
  } else if constexpr (G == KG_WIDE) {
    switch (st) {
      case ZK_ES_SHL_SHR: gadget_shl_shr(s, true); break;
      default: break;
    }
  } else if constexpr (G == KG_TX) {
    switch (st) {
      case ZK_ES_STOP: gadget_stop(s, true); break;
      case ZK_ES_BeginTx: gadget_begin_tx(s, (flags & ZK_FLAG_EVM_FIRST_STEP) && s.row == 0); break;
      case ZK_ES_EndTx: gadget_end_tx(s); break;
      case ZK_ES_EndBlock: gadget_end_block(s, (flags & ZK_FLAG_EVM_LAST_STEP) && s.i == s.w.n_rows - 2); break;
      case ZK_ES_ErrorStack: gadget_error_stack(s); break;
      case ZK_ES_ErrorInvalidOpcode: gadget_error_invalid_opcode(s); break;
      case ZK_ES_ErrorOutOfGasConstant: gadget_error_oog_constant(s); break;
      case ZK_ES_ErrorInvalidJump: gadget_error_invalid_jump(s); break;
      case ZK_ES_SELFBALANCE: gadget_selfbalance(s); break;
      case ZK_ES_ErrorOutOfGasSHA3: gadget_error_oog_sha3(s); break;
      case ZK_ES_ErrorOutOfGasStaticMemoryExpansion: gadget_error_oog_static_memory(s); break;
      case ZK_ES_ErrorOutOfGasDynamicMemoryExpansion: gadget_error_oog_dynamic_memory(s); break;
      case ZK_ES_ErrorOutOfGasLOG: gadget_error_oog_log(s); break;
      case ZK_ES_ErrorOutOfGasEXP: gadget_error_oog_exp(s); break;
      case ZK_ES_ErrorReturnDataOutOfBound: gadget_error_return_data_oob(s); break;
      case ZK_ES_BALANCE: gadget_account_access(s, 0x31); break;
      case ZK_ES_EXTCODEHASH: gadget_account_access(s, 0x3f); break;
      case ZK_ES_EXTCODESIZE: gadget_account_access(s, 0x3b); break;
      case ZK_ES_ErrorOutOfGasAccountAccess: gadget_error_oog_account_access(s); break;
      case ZK_ES_CODECOPY: gadget_codecopy(s); break;
      case ZK_ES_RETURNDATACOPY: gadget_returndatacopy(s); break;
      case ZK_ES_EXTCODECOPY: gadget_extcodecopy(s); break;
      case ZK_ES_ErrorOutOfGasMemoryCopy: gadget_error_oog_memory_copy(s); break;
      case ZK_ES_SLOAD: gadget_sload(s); break;
      case ZK_ES_SSTORE: gadget_sstore(s); break;
      case ZK_ES_CALLDATALOAD: gadget_calldataload(s); break;
      case ZK_ES_LOG: gadget_log(s); break;
      case ZK_ES_ErrorWriteProtection: gadget_error_write_protection(s); break;
      case ZK_ES_BLOCKHASH: gadget_blockhash(s); break;
      case ZK_ES_ErrorMaxCodeSizeExceeded: case ZK_ES_ErrorOutOfGasCodeStore: gadget_error_code_store(s); break;
      case ZK_ES_ErrorInvalidCreationCode: gadget_error_invalid_creation_code(s); break;
      case ZK_ES_RETURN: gadget_return_revert(s); break;
      case ZK_ES_ErrorOutOfGasCall: gadget_error_oog_call(s); break;
      case ZK_ES_CALL_OP: gadget_callop(s); break;
      case ZK_ES_CREATE: case ZK_ES_CREATE2: gadget_create(s); break;
      case ZK_ES_ErrorOutOfGasSloadSstore: gadget_error_oog_sload_sstore(s); break;
      case ZK_ES_ErrorOutOfGasCREATE: gadget_error_oog_create(s); break;
      case ZK_ES_ErrorOutOfGasPrecompile: gadget_error_oog_precompile(s); break;
      case ZK_ES_ErrorGasUintOverflow: gadget_error_gas_uint_overflow(s); break;
      default: break;
    }
  } else if constexpr (G == KG_ARITH) {
    switch (st) {
      case ZK_ES_ADDMOD: gadget_addmod_mulmod(s, false); break;
      case ZK_ES_MULMOD: gadget_addmod_mulmod(s, true); break;
      case ZK_ES_SDIV_SMOD: gadget_sdiv_smod(s); break;
      case ZK_ES_SAR: gadget_sar(s); break;
      case ZK_ES_EXP: gadget_exp(s); break;
      default: break;
    }
  }
}

// whole step on one thread (tests/emu)
ZK_HD void verify_step(const StepCtx& s, u32 flags) {
  const int st = step_prologue(s, flags);
  if (st < 0) return;
  switch (es_group(st)) {
    case KG_ADD: gadget_add(s, true); break;
    case KG_MUL: gadget_mul(s, true); break;
    case KG_PUSH:
      if (both_positional(s.t)) {  // what k_evm_push_pos runs
        HeadCache hc{};
        gadget_push_pos1(s, &hc);
      } else {
        gadget_push(s, true);
      }
      break;
    case KG_POP: gadget_pop(s, true); break;
    case KG_SIMPLE: run_group<KG_SIMPLE>(s, st, flags); break;
    case KG_BYTES32: run_group<KG_BYTES32>(s, st, flags); break;
    case KG_COPY: run_group<KG_COPY>(s, st, flags); break;
    case KG_WIDE: run_group<KG_WIDE>(s, st, flags); break;
    case KG_TX: run_group<KG_TX>(s, st, flags); break;
    case KG_ARITH: run_group<KG_ARITH>(s, st, flags); break;
    default: break;
  }
}

// ======================================================================================
// kernels
// ======================================================================================
// The reference dispatches one Python gadget per step (execution/__init__.py:86-171).  Here the steps
// are SORTED by execution state first — k_evm_classify runs the cheap prologue of every step, writes
// its bucket and a histogram; k_evm_scatter turns the histogram into bucket offsets and writes the
// step indices bucket by bucket (a counting sort, one byte + one u32 per step) — and then one kernel
// per gate-program group walks its buckets, so the lanes of a warp run the same straight-line program.
struct EvmSort {
  unsigned char* bucket;  // [n] bucket of local step k (ZK_BK_NONE: it failed in the prologue)
  u32* hist;              // [ZK_EVM_NB + 1] steps per bucket (entry ZK_EVM_NB unused)
  u32* cursor;            // [ZK_EVM_NB] scatter cursors (zeroed by the host)
  u32* offs;              // [ZK_EVM_NB + 1] first entry of each bucket in `sorted`
  u32* sorted;            // [n] local step indices, bucket by bucket
};

// Table-derived constants of EndBlock (end_block.py:68-105).  The reference's tables are Python sets, so a
// row identical in every column to an earlier one does not count.
ZK_HD bool first_of_kind_ix(const IndexDev& ix, u32 r) {  // via the table's hash index: no identical row before r
  const TableDev& t = ix.tab;
  Fr h = table_cell(t, ix.key_cols[0], r);
  for (u32 j = 1; j < ix.n_key; j++) h = fr_add(h, rlc_term(ix, table_cell(t, ix.key_cols[j], r), (int)j));
  const u64 mix = rlc_mix(h);
  const u32 fp = (u32)(mix >> 32);
  u32 b = (u32)mix & ix.mask;
  for (;;) {
    const u64 slot = ld_u64(&ix.slots[b]);
    if (slot == ZK_EMPTY_SLOT) return true;
    const u32 cand = (u32)slot;
    if ((u32)(slot >> 32) == fp && cand < r && rows_identical(t, cand, r)) return false;
    b = (b + 1) & ix.mask;
  }
}
ZK_HD void block_stats_tx_row(const IndexDev& tx, u32 r, BlockStats* out) {
  const Fr tag = table_cell(tx.tab, 1, r);
  const bool caller = fr_eq_u64(tag, ZK_TX_CallerAddress), invalid = fr_eq_u64(tag, ZK_TX_TxInvalid);
  if (!(caller || invalid) || !first_of_kind_ix(tx, r)) return;
  const Fr lo = table_cell(tx.tab, 3, r), hi = table_cell(tx.tab, 4, r);
  if (caller) {
    atomic_add_u32(&out->max_txs, 1);
    if (!(fr_is_zero(lo) && fr_is_zero(hi))) atomic_add_u32(&out->total_txs, 1);
  } else {
    if (tx.tab.flags && (tx.tab.flags[r] & 1)) atomic_add_u32(&out->txinvalid_word, 1);
    else if (fr_eq_u64(lo, 1)) atomic_add_u32(&out->invalid_txs, 1);
  }
}
ZK_HD void block_stats_wd_row(const TableDev& wd, u32 r, BlockStats* out) {
  for (u32 q = 0; q < r; q++)
    if (rows_identical(wd, q, r)) return;
  atomic_add_u32(&out->max_wds, 1);
  if (!fr_is_zero(table_cell(wd, 3, r))) atomic_add_u32(&out->total_wds, 1);
}

#ifdef __CUDACC__
// one thread per row of the largest of the three tables; `rw_rwc` may be unbuilt when the rw table is dense
__global__ void __launch_bounds__(256) k_evm_block_stats(EvmTables t, BlockStats* out) {
  const u64 stride = (u64)gridDim.x * blockDim.x, tid = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  for (u64 r = tid; r < t.tx.tab.n_rows; r += stride) block_stats_tx_row(t.tx, (u32)r, out);
  for (u64 r = tid; r < t.wd.n_rows; r += stride) block_stats_wd_row(t.wd, (u32)r, out);
  if (pos_enabled(t.rw) && t.rw.pos_kind == ZK_POS_DENSE) {  // distinct counters: every row is its own kind
    if (tid == 0) out->max_rws = (u32)t.rw.tab.n_rows;
  } else {
    for (u64 r = tid; r < t.rw.tab.n_rows; r += stride)
      if (first_of_kind_ix(t.rw_rwc, (u32)r)) atomic_add_u32(&out->max_rws, 1);
  }
}

// MUL-state steps are split three ways by an UNVERIFIED peek at their opcode (positional tables only):
// MUL, DIV and MOD take three different witness-assignment branches (mul_div_mod.py:23-41), and a warp
// that holds all three runs them one after the other.  The peek only chooses the bucket — the gate
// program looks the opcode up again and decides everything itself — so a wrong peek costs time, never
// the verdict.
__device__ __forceinline__ int mul_bucket_peek(const StepCtx& s, const Fr& hlo, const Fr& hhi, const Fr& pc) {
  u32 head = 0, len = 0;
  if (heads_probe(s.t.bytecode, hlo, hhi, &head, &len, s.mask, true) != 1) return ZK_ES_MUL;
  if (!(fr_fits64(pc) && pc.l[0] < (u64)len)) return ZK_ES_MUL;
  const Fr v = table_cell(s.t.bytecode.tab, B_VALUE, (u64)head + 1 + pc.l[0]);
  return fr_eq_u64(v, 4) ? ZK_BK_DIV : (fr_eq_u64(v, 6) ? ZK_BK_MOD : ZK_ES_MUL);
}

// NARROW: StepCtx::narrow (the step cells but the code hash sit in columns of at most 8 bytes: one aligned load each)
template <int NARROW>
__global__ void __launch_bounds__(1024) k_evm_classify(const __grid_constant__ WitnessDev w, const __grid_constant__ CheckRange rg, const __grid_constant__ EvmTables t, const __grid_constant__ ResultDev res, const __grid_constant__ EvmSort so) {
  // histogram aggregated per BLOCK: lanes of a warp that share a bucket elect a leader (match_any),
  // leaders add to a shared histogram, one global atomicAdd per (block, non-empty bucket)
  __shared__ u32 s_hist[ZK_EVM_NB];
  if (threadIdx.x < ZK_EVM_NB) s_hist[threadIdx.x] = 0;
  __syncthreads();
  const u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  const u64 i = rg.row_begin + k;
  const unsigned lane = threadIdx.x & 31;
  // the peek needs the bytecode table's heads index alone; the rw index may still be verifying on another stream
  // (check_evm), so its flag is not read here
  const bool pos = t.bytecode.tab.n_rows != 0 && pos_enabled(t.bytecode) && t.bytecode.pos_kind == ZK_POS_RUNS;
  int b = ZK_BK_NONE;
  if (i < rg.row_end) {
    StepCtx s{w, t, res, i, i + 1, rg.row_base + i, true, nullptr, 1u << lane, nullptr, nullptr, -1, NARROW};
    // the peek's cells are fetched with the state cells (one memory round trip instead of two)
    const Fr hlo = s.cur(S_HASH_LO), hhi = s.cur(S_HASH_HI), pc = s.cur(S_PC);
    const int st = step_prologue(s, rg.flags);
    if (st >= 0) b = (st == ZK_ES_MUL && pos) ? mul_bucket_peek(s, hlo, hhi, pc) : st;
    so.bucket[k] = (unsigned char)b;
  }
  const unsigned m = __match_any_sync(0xFFFFFFFFu, b);
  if (b != ZK_BK_NONE && lane == (unsigned)(__ffs(m) - 1)) atomicAdd(&s_hist[b], (u32)__popc(m));
  __syncthreads();
  if (threadIdx.x < ZK_EVM_NB && s_hist[threadIdx.x]) atomicAdd(&so.hist[threadIdx.x], s_hist[threadIdx.x]);
}

__global__ void __launch_bounds__(1024) k_evm_scatter(EvmSort so, u32 n) {
  __shared__ u32 s_off[ZK_EVM_NB + 1], s_cnt[ZK_EVM_NB], s_base[ZK_EVM_NB], s_wsum[ZK_EVM_NB / 32];
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x < ZK_EVM_NB) {  // exclusive scan of the histogram (4 warps)
    const u32 c = so.hist[threadIdx.x];
    u32 v = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const u32 u = __shfl_up_sync(0xFFFFFFFFu, v, d);
      if ((int)lane >= d) v += u;
    }
    if (lane == 31) s_wsum[warp] = v;
    s_off[threadIdx.x] = v - c;
    s_cnt[threadIdx.x] = 0;
  }
  __syncthreads();
  if (threadIdx.x < ZK_EVM_NB) {
    u32 add = 0;
    for (unsigned q = 0; q < warp; q++) add += s_wsum[q];
    s_off[threadIdx.x] += add;
    if (threadIdx.x == ZK_EVM_NB - 1) s_off[ZK_EVM_NB] = s_off[threadIdx.x] + so.hist[threadIdx.x];
  }
  const u32 k = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = k < n ? (int)so.bucket[k] : ZK_BK_NONE;
  const unsigned m = __match_any_sync(0xFFFFFFFFu, b);
  const int leader = __ffs(m) - 1;
  const u32 rank = __popc(m & ((1u << lane) - 1));
  __syncthreads();
  u32 wbase = 0;
  if (b != ZK_BK_NONE && (int)lane == leader) wbase = atomicAdd(&s_cnt[b], (u32)__popc(m));
  wbase = __shfl_sync(0xFFFFFFFFu, wbase, leader);
  __syncthreads();
  if (threadIdx.x < ZK_EVM_NB && s_cnt[threadIdx.x]) s_base[threadIdx.x] = atomicAdd(&so.cursor[threadIdx.x], s_cnt[threadIdx.x]);
  __syncthreads();
  if (b != ZK_BK_NONE) so.sorted[s_off[b] + s_base[b] + wbase + rank] = k;
  if (blockIdx.x == 0 && threadIdx.x <= ZK_EVM_NB) so.offs[threadIdx.x] = s_off[threadIdx.x];
}

// one thread per step for the gadgets whose work is a handful of independent lookups.
// POS = both tables positional (known to the host from the read-back flag): that instance is compiled
// with pos_mode = 1, i.e. without any hash-index code — these kernels were stalling on instruction
// fetch (profiles/README.md v20: "no instruction" 2-3 per issue), the executed path is now half as long.
// POS: 0 = hash indexes, 1 = both tables positional, 2 = positional AND narrow (StepCtx::narrow)
template <int G, int POS>
__device__ __forceinline__ void bucket_steps(const WitnessDev& w, const CheckRange& rg, const EvmTables& t,
                                             const ResultDev& res, const EvmSort& so, const u32* s_resp, int bucket,
                                             const Fr* stack_pre, const u64& rw_base) {
  // every lane of a warp runs the same number of rounds and calls the (warp-synchronous) lookups
  // together; lanes without a step in the last round run with live = false
  const u32 n = so.hist[bucket];
  if (n == 0) return;
  const u32* list = so.sorted + so.offs[bucket];
  const u32 stride = gridDim.x * blockDim.x;
  const u32 tid = blockIdx.x * blockDim.x + threadIdx.x;
  for (u32 first = 0; first < n; first += stride) {
    const u32 k = first + tid;
    const bool live = k < n;
    const u64 i = rg.row_begin + list[live ? k : 0];
    StepCtx s{w, t, res, i, i + 1, rg.row_base + i, live, s_resp, 0xFFFFFFFFu, POS ? nullptr : stack_pre,
              POS ? &rw_base : nullptr, POS ? 1 : -1, POS == 2 ? 1 : 0};
    if (G == KG_ADD) gadget_add(s, live);
    else if (G == KG_MUL) gadget_mul(s, live);
    else gadget_pop(s, live);
  }
}
// minimum resident blocks per SM (= register caps of 168 / 128): measured sweep in
// profiles/r01_v25_launch_bounds_sweep.json — (3, 4) cuts the check phase from 0.539 to 0.443 ms
#ifndef ZK_GADGET_MINBLOCKS
#define ZK_GADGET_MINBLOCKS 3
#endif
#ifndef ZK_PUSH_MINBLOCKS
#define ZK_PUSH_MINBLOCKS 4
#endif
// ADD / SUB and POP are latency-bound on three dependent round trips (8-9 long-scoreboard stalls per issue,
// profiles/r02_m_top_kernels_ncu_full.csv): 6 resident blocks (80 registers; POP without a spill, ADD with 216 bytes)
// beat 3 (142 / 107 registers) by 3 % of the check phase (profiles/r02_m_launch_bound_variants.json)
#ifndef ZK_ADD_MINBLOCKS
#define ZK_ADD_MINBLOCKS 6
#endif
#ifndef ZK_POP_MINBLOCKS
#define ZK_POP_MINBLOCKS 6
#endif
template <int G, int POS>
__global__ void __launch_bounds__(128, G == KG_MUL ? ZK_GADGET_MINBLOCKS : (G == KG_ADD ? ZK_ADD_MINBLOCKS : ZK_POP_MINBLOCKS))
k_evm_gadget(const __grid_constant__ WitnessDev w, const __grid_constant__ CheckRange rg, const __grid_constant__ EvmTables t, const __grid_constant__ ResultDev res,
             const __grid_constant__ EvmSort so) {
  __shared__ alignas(16) u32 s_resp[ZK_RESP_BITMAP_WORDS];
  __shared__ alignas(8) u64 s_bar;
  stage_to_smem(s_resp, t.resp_bitmap, sizeof(s_resp), &s_bar);
  Fr stack_pre[2];
  if (!POS) stack_key_pre(t.rw, stack_pre);
  const u64 rw_base = POS ? table_cell(t.rw.tab, 0, 0).l[0] : 0;
  if (G == KG_MUL) {  // three buckets (opcode peeks MUL / DIV / MOD), one after the other: warps stay uniform
#pragma unroll 1
    for (int sub = 0; sub < 3; sub++)
      bucket_steps<G, POS>(w, rg, t, res, so, s_resp, sub == 0 ? ZK_ES_MUL : (sub == 1 ? ZK_BK_DIV : ZK_BK_MOD), stack_pre, rw_base);
  } else {
    bucket_steps<G, POS>(w, rg, t, res, so, s_resp, G == KG_ADD ? ZK_ES_ADD : ZK_ES_POP, stack_pre, rw_base);
  }
}

// rare groups: a thread takes one step of one bucket at a time; a warp may straddle two buckets at a
// bucket boundary, so every lookup is lane-private (mask = the lane's own bit: the probe loops need
// no warp agreement)
template <int G>
__global__ void __launch_bounds__(128) k_evm_group(const __grid_constant__ WitnessDev w, const __grid_constant__ CheckRange rg,
                                                   const __grid_constant__ EvmTables t, const __grid_constant__ ResultDev res,
                                                   const __grid_constant__ EvmSort so) {
  // __grid_constant__: the out-of-line lookups take these structures by reference; without it every
  // thread first copies the 12 KB of kernel parameters to its local-memory stack
  __shared__ alignas(16) u32 s_resp[ZK_RESP_BITMAP_WORDS];
  __shared__ alignas(8) u64 s_bar;
  stage_to_smem(s_resp, t.resp_bitmap, sizeof(s_resp), &s_bar);
  const u32 stride = gridDim.x * blockDim.x;
#pragma unroll 1
  for (int st = 0; st < ZK_ES_COUNT; st++) {
    if (es_group(st) != G) continue;
    const u32 n = so.hist[st];
    if (n == 0) continue;
    const u32* list = so.sorted + so.offs[st];
    for (u32 k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride) {
      const u64 i = rg.row_begin + list[k];
      StepCtx s{w, t, res, i, i + 1, rg.row_base + i, true, s_resp, 1u << (threadIdx.x & 31), nullptr, nullptr, -1};
      run_group<G>(s, st, rg.flags);
    }
  }
}

__device__ __forceinline__ Fr shfl_fr(const Fr& v, int src) {
  Fr r;
#pragma unroll
  for (int k = 0; k < 4; k++) r.l[k] = __shfl_sync(0xFFFFFFFFu, v.l[k], src);
  return r;
}
__device__ __forceinline__ Fr shfl16_fr(const Fr& v, int src) {
  Fr r;
#pragma unroll
  for (int k = 0; k < 4; k++) r.l[k] = __shfl_sync(0xFFFFFFFFu, v.l[k], src, 16);
  return r;
}
// positional rw + bytecode tables: one thread per PUSH step (gadget_push_pos1); NARROW: StepCtx::narrow
template <int NARROW>
__global__ void __launch_bounds__(128, ZK_PUSH_MINBLOCKS) k_evm_push_pos(const __grid_constant__ WitnessDev w, const __grid_constant__ CheckRange rg, const __grid_constant__ EvmTables t, const __grid_constant__ ResultDev res,
               const __grid_constant__ EvmSort so) {
  __shared__ alignas(16) u32 s_resp[ZK_RESP_BITMAP_WORDS];
  __shared__ alignas(8) u64 s_bar;
  stage_to_smem(s_resp, t.resp_bitmap, sizeof(s_resp), &s_bar);
  const u64 rw_base = table_cell(t.rw.tab, 0, 0).l[0];
  HeadCache hc{};
  const u32 n = so.hist[ZK_ES_PUSH];
  const u32* list = so.sorted + so.offs[ZK_ES_PUSH];
  const u32 stride = gridDim.x * blockDim.x;
  for (u32 k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride) {
    const u64 i = rg.row_begin + list[k];
    StepCtx s{w, t, res, i, i + 1, rg.row_base + i, true, s_resp, 1u << (threadIdx.x & 31), nullptr, &rw_base, 1, NARROW};
    gadget_push_pos1(s, &hc);
  }
}

// The generic path (tables not positional).  Half a warp per PUSH step (two steps per warp
// iteration): sub-lane L of a half owns pushed bytes L and L+16 of its step, so the warp-synchronous
// hash probes of a step's 34 bytecode lookups run side by side.  Halving the lanes per step halves
// the warp-instructions per step and doubles the steps in flight per warp; the kernel is
// latency-bound on ~8 dependent memory round trips per step (profiles/README.md, v7).  All 32 lanes
// call every warp-synchronous lookup together; a half without a step (odd count) or whose step
// already failed passes live = false.
__global__ void __launch_bounds__(128, 4) k_evm_push_hash(const __grid_constant__ WitnessDev w, const __grid_constant__ CheckRange rg, const __grid_constant__ EvmTables t, const __grid_constant__ ResultDev res,
                const __grid_constant__ EvmSort so) {
  __shared__ alignas(16) u32 s_resp[ZK_RESP_BITMAP_WORDS];
  __shared__ alignas(8) u64 s_bar;
  stage_to_smem(s_resp, t.resp_bitmap, sizeof(s_resp), &s_bar);
  Fr stack_pre[2];
  stack_key_pre(t.rw, stack_pre);
  Fr last_hlo = fr_u64(0), last_hhi = fr_u64(0), last_h0 = fr_u64(0);  // per-lane cache of the last code hash seen
  bool have_h0 = false;
  const u32 n = so.hist[ZK_ES_PUSH];
  const u32* list = so.sorted + so.offs[ZK_ES_PUSH];
  const int lane = threadIdx.x & 31, half = lane >> 4, sub = lane & 15;
  const u32 warps = (gridDim.x * blockDim.x) >> 5;
  const u32 n_pairs = (n + 1) >> 1;
  const int kNone = 0x7FFFFFFF;
  for (u32 kp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; kp < n_pairs; kp += warps) {  // warp-uniform
    const u32 k = 2 * kp + half;
    const bool have = k < n;
    bool live = have;
    const u64 i = rg.row_begin + list[have ? k : 2 * kp];
    StepCtx s{w, t, res, i, i + 1, rg.row_base + i, have && sub == 0, s_resp, 0xFFFFFFFFu, stack_pre, nullptr, -1};
    PushCommon c;
    c.hlo = s.cur(S_HASH_LO);
    c.hhi = s.cur(S_HASH_HI);
    c.pc = s.cur(S_PC);
    // this lane's cell of the current / next step for the epilogue, fetched with the first batch
    const Fr my_cur = s.cur((u32)(sub < 13 ? sub : 0)), my_nxt = s.nxt((u32)(sub < 13 ? sub : 0));
    // consecutive steps of a lane almost always run the same contract: reuse the work that depends
    // only on the code hash (hash_lo + hash_hi*r; with positional tables, the run head itself)
    const bool changed = !(have_h0 && fr_eq(c.hlo, last_hlo) && fr_eq(c.hhi, last_hhi));
    if (changed) {
      last_hlo = c.hlo;
      last_hhi = c.hhi;
      last_h0 = bytecode_hash0(s, c.hlo, c.hhi);
      have_h0 = true;
    }
    c.h0 = last_h0;
    // (one of the two tables may still be positional: bytecode_head / the lookups below test the flags)
    c.n_head = bytecode_head(s, live, c.hlo, c.hhi, &c.head, &c.run_len);
    // round 1: sub-lane 0 opcode, 1 bytecode length (one warp-wide bytecode probe), then sub-lane 2
    // the stack_push row (one warp-wide rw probe)
    Fr v = fr_u64(0);
    Word2 val{fr_u64(0), fr_u64(0)};
    int n_hit = bytecode_lookup_h(s, live && sub < 2, c.h0, c.n_head, c.head, c.run_len, c.hlo, c.hhi, sub == 0 ? 2 : 1,
                                  sub == 0 ? c.pc : fr_u64(0), sub == 0 ? 1 : 0, &v);
    const int n_hit_rw = rw_lookup(s, live && sub == 2, s.cur(S_RWC), 1, ZK_TARGET_Stack, s.cur(S_CALL_ID),
                                   fr_sub_u64(s.cur(S_SP), 1), &val);
    if (sub == 2) n_hit = n_hit_rw;
    const int n_op = __shfl_sync(0xFFFFFFFFu, n_hit, 0, 16), n_len = __shfl_sync(0xFFFFFFFFu, n_hit, 1, 16);
    const int n_rw = __shfl_sync(0xFFFFFFFFu, n_hit, 2, 16);
    const Fr opcode = shfl16_fr(v, 0), code_length = shfl16_fr(v, 1);
    Word2 value{shfl16_fr(val.lo, 2), shfl16_fr(val.hi, 2)};
    if (live) live = push_prepare(s, n_op, opcode, n_len, code_length, n_rw, value, &c);  // uniform per half
    // round 2: pushed bytes L and L+16; the first failing byte in program order wins
    const int fid0 = push_byte(s, c, sub, live), fid1 = push_byte(s, c, sub + 16, live);
    const unsigned bad0 = (__ballot_sync(0xFFFFFFFFu, live && fid0 >= 0) >> (16 * half)) & 0xFFFFu;
    const unsigned bad1 = (__ballot_sync(0xFFFFFFFFu, live && fid1 >= 0) >> (16 * half)) & 0xFFFFu;
    if (bad0) {
      if (sub == __ffs(bad0) - 1) fail(res, fid0, s.row);
      live = false;
    } else if (bad1) {
      if (sub == __ffs(bad1) - 1) fail(res, fid1, s.row);
      live = false;
    }
    int eid = kNone;
    if (live) eid = same_context_lane(s, sub, my_cur, my_nxt, c.opcode, 1, fr_add_u64(c.num_pushed, 1), fr_sub(fr_u64(0), fr_u64(1)));
#pragma unroll
    for (int off = 8; off >= 1; off >>= 1) eid = min(eid, __shfl_xor_sync(0xFFFFFFFFu, eid, off, 16));
    if (live && eid != kNone && sub == 0) fail(res, eid, s.row);
  }
}
#endif  // __CUDACC__

}  // namespace zk
