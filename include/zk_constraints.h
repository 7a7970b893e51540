/*
 * zk_constraints.h — constraint catalogue: the ids that index first_fail[] / fail_count[].
 *
 * Ids are numbered in the reference's PROGRAM ORDER inside one row / step, so that
 * "the exception the reference raises first" == the failing id with the smallest
 * (row, id) pair.  X(id_name, error_class, "reference file:line — what it asserts").
 * Both the CUDA product and the CPU oracle include this file; it contains no code.
 */
#ifndef ZK_CONSTRAINTS_H
#define ZK_CONSTRAINTS_H

/* error classes mirror ZK_ERR_* in zkcheck.h */
#define ZKE_ASSERT 0
#define ZKE_UNSAT 1
#define ZKE_AMBIG 2
#define ZKE_RANGE 3
#define ZKE_VALUE 4
#define ZKE_NOTIMPL 5

/* ---------------- bytecode circuit: src/zkevm_specs/bytecode_circuit.py:37-100 ------- */
#define ZK_BYTECODE_CONSTRAINTS(X)                                                        \
  X(BC_FIRST_TAG, ZKE_ASSERT, "bytecode_circuit.py:44-45 q_first => tag==Header")         \
  X(BC_HDR_VALUE_LEN, ZKE_ASSERT, "bytecode_circuit.py:49 header value==length")          \
  X(BC_HDR_INDEX0, ZKE_ASSERT, "bytecode_circuit.py:50 header index==0")                  \
  X(BC_H2B_LEN, ZKE_ASSERT, "bytecode_circuit.py:73 next.length==length")                 \
  X(BC_H2B_INDEX0, ZKE_ASSERT, "bytecode_circuit.py:74 next.index==0")                    \
  X(BC_H2B_ISCODE, ZKE_ASSERT, "bytecode_circuit.py:75 next.is_code==1")                  \
  X(BC_H2B_HASH, ZKE_ASSERT, "bytecode_circuit.py:76 next.hash==hash")                    \
  X(BC_H2B_RLC, ZKE_ASSERT, "bytecode_circuit.py:77 next.value_rlc==next.value")          \
  X(BC_H2H_LEN0, ZKE_ASSERT, "bytecode_circuit.py:81 length==0")                          \
  X(BC_H2H_EMPTY_HASH, ZKE_ASSERT, "bytecode_circuit.py:82 hash==EMPTY_HASH")             \
  X(BC_PUSH_TABLE, ZKE_ASSERT, "bytecode_circuit.py:57 (value,push_data_size) in push_table") \
  X(BC_IS_CODE, ZKE_ASSERT, "bytecode_circuit.py:58 is_code==(push_data_left==0)")        \
  X(BC_B2B_LEN, ZKE_ASSERT, "bytecode_circuit.py:87 next.length==length")                 \
  X(BC_B2B_INDEX, ZKE_ASSERT, "bytecode_circuit.py:88 next.index==index+1")               \
  X(BC_B2B_HASH, ZKE_ASSERT, "bytecode_circuit.py:89 next.hash==hash")                    \
  X(BC_B2B_RLC, ZKE_ASSERT, "bytecode_circuit.py:90 next.value_rlc==value_rlc*r+next.value") \
  X(BC_B2B_PUSH_LEFT, ZKE_ASSERT, "bytecode_circuit.py:91-94 push_data_left transition")  \
  X(BC_B2H_INDEX, ZKE_ASSERT, "bytecode_circuit.py:99 index+1==length")                   \
  X(BC_B2H_KECCAK, ZKE_ASSERT, "bytecode_circuit.py:100 (2,value_rlc,length,hash) in keccak_table") \
  X(BC_LAST_TAG, ZKE_ASSERT, "bytecode_circuit.py:66 q_last => tag==Header")              \
  X(BC_LAST_LEN0, ZKE_ASSERT, "bytecode_circuit.py:67,81 q_last => length==0")            \
  X(BC_LAST_EMPTY_HASH, ZKE_ASSERT, "bytecode_circuit.py:67,82 q_last => hash==EMPTY_HASH")

/* generic enum builder */
#define ZK_ENUM_ENTRY(id, cls, doc) id,

enum zk_bytecode_constraint { ZK_BYTECODE_CONSTRAINTS(ZK_ENUM_ENTRY) BC_N_CONSTRAINTS };

/* ---------------- EVM circuit: src/zkevm_specs/evm_circuit/main.py:47-63 and the gadgets ----
 * One step runs: the common prologue, exactly one gadget block, and (for same-context
 * opcodes) the shared epilogue EV_SC_*; ids inside each block follow program order. */
#define ZK_EVM_PUSH_BYTE(X, i)                                                              \
  X(EV_PUSH_B##i##_UNSAT, ZKE_UNSAT, "push.py:25-27 byte " #i ": bytecode lookup (is_code=0) unsat")  \
  X(EV_PUSH_B##i##_AMBIG, ZKE_AMBIG, "push.py:25-27 byte " #i ": bytecode lookup ambiguous")          \
  X(EV_PUSH_B##i##_EQ, ZKE_ASSERT, "push.py:25-27 byte " #i ": pushed byte == bytecode byte")        \
  X(EV_PUSH_B##i##_ZERO, ZKE_ASSERT, "push.py:29 byte " #i ": unpushed/padding byte == 0")

#define ZK_EVM_RESTORE_LOOKUP(X, k)                                                          \
  X(EV_RST##k##_UNSAT, ZKE_UNSAT, "instruction.py:304-336 restore-context lookup " #k " unsat")      \
  X(EV_RST##k##_AMBIG, ZKE_AMBIG, "instruction.py:304-336 restore-context lookup " #k " ambiguous")  \
  X(EV_RST##k##_CHECK, ZKE_ASSERT, "instruction.py:304-336 restore-context lookup " #k ": .value() type / written value")

#define ZK_EVM_CONSTRAINTS(X)                                                               \
  X(EV_FIRST_STATE, ZKE_ASSERT, "main.py:48-52 first step state in {BeginTx,EndBlock}")     \
  X(EV_FIRST_RWC, ZKE_ASSERT, "main.py:53 first step rw_counter==1")                        \
  X(EV_LAST_STATE, ZKE_ASSERT, "main.py:55-56 last step state==EndBlock")                   \
  X(EV_TRANS_FROM_ENDTX, ZKE_ASSERT, "instruction.py:193-194 EndTx -> BeginTx|EndBlock")    \
  X(EV_TRANS_FROM_ENDBLOCK, ZKE_ASSERT, "instruction.py:195-196 EndBlock -> EndBlock")      \
  X(EV_TRANS_TO_BEGINTX, ZKE_ASSERT, "instruction.py:199-200 -> BeginTx only from EndTx")   \
  X(EV_TRANS_TO_ENDTX, ZKE_ASSERT, "instruction.py:201-202 -> EndTx only from halting|BeginTx") \
  X(EV_TRANS_TO_ENDBLOCK, ZKE_ASSERT, "instruction.py:203-204 -> EndBlock only from EndTx|EndBlock") \
  X(EV_NOT_IMPLEMENTED, ZKE_NOTIMPL, "main.py:60-63 state has no gadget in the reference")  \
  X(EV_UNSUPPORTED_STATE, ZKE_NOTIMPL, "this build has no gate program for the state")      \
  X(EV_OP_UNSAT, ZKE_UNSAT, "instruction.py:784-790 opcode_lookup: bytecode lookup unsat")  \
  X(EV_OP_AMBIG, ZKE_AMBIG, "instruction.py:784-790 opcode_lookup: bytecode lookup ambiguous") \
  /* ADD / SUB: execution/add_sub.py:5-24 */                                                \
  X(EV_ADD_A_UNSAT, ZKE_UNSAT, "add_sub.py:10 stack_pop a unsat")                           \
  X(EV_ADD_A_AMBIG, ZKE_AMBIG, "add_sub.py:10 stack_pop a ambiguous")                       \
  X(EV_ADD_B_UNSAT, ZKE_UNSAT, "add_sub.py:11 stack_pop b unsat")                           \
  X(EV_ADD_B_AMBIG, ZKE_AMBIG, "add_sub.py:11 stack_pop b ambiguous")                       \
  X(EV_ADD_C_UNSAT, ZKE_UNSAT, "add_sub.py:12 stack_push c unsat")                          \
  X(EV_ADD_C_AMBIG, ZKE_AMBIG, "add_sub.py:12 stack_push c ambiguous")                      \
  X(EV_ADD_SUM, ZKE_ASSERT, "add_sub.py:14-17 add_words([is_sub?c:a, b]) == (is_sub?a:c)")   \
  /* MUL / DIV / MOD: execution/mul_div_mod.py:6-71 */                                      \
  X(EV_MUL_POP1_UNSAT, ZKE_UNSAT, "mul_div_mod.py:18 stack_pop unsat")                      \
  X(EV_MUL_POP1_AMBIG, ZKE_AMBIG, "mul_div_mod.py:18 stack_pop ambiguous")                  \
  X(EV_MUL_POP2_UNSAT, ZKE_UNSAT, "mul_div_mod.py:19 stack_pop unsat")                      \
  X(EV_MUL_POP2_AMBIG, ZKE_AMBIG, "mul_div_mod.py:19 stack_pop ambiguous")                  \
  X(EV_MUL_PUSH_UNSAT, ZKE_UNSAT, "mul_div_mod.py:20 stack_push unsat")                     \
  X(EV_MUL_PUSH_AMBIG, ZKE_AMBIG, "mul_div_mod.py:20 stack_push ambiguous")                 \
  X(EV_MUL_WITNESS_DOMAIN, ZKE_NOTIMPL, "DIV/MOD witness assignment with a stack word half >= 2^128: outside the supported witness domain (DESIGN.md)") \
  X(EV_MUL_WITNESS_NEG, ZKE_VALUE, "mul_div_mod.py:32,41 Word(negative int) -> OverflowError") \
  X(EV_MUL_TO64, ZKE_VALUE, "instruction.py:604-605 to_64s(): half of a or b >= 2^128 -> OverflowError") \
  X(EV_MUL_CARRY_LO, ZKE_RANGE, "instruction.py:626 range_check(carry_lo, 9)")              \
  X(EV_MUL_CARRY_HI, ZKE_RANGE, "instruction.py:627 range_check(carry_hi, 9)")              \
  X(EV_MUL_SELECT, ZKE_ASSERT, "mul_div_mod.py:47-54 select_word bool / Word range asserts") \
  X(EV_MUL_PUSH_EQ, ZKE_ASSERT, "mul_div_mod.py:49-54 push == d*is_mul + a*is_div*(1-b0) + c*is_mod*(1-b0)") \
  X(EV_MUL_C_ZERO, ZKE_ASSERT, "mul_div_mod.py:57 is_mul * sum(bytes(c)) == 0")             \
  X(EV_MUL_REM_LT, ZKE_ASSERT, "mul_div_mod.py:60-61 remainder < divisor unless divisor==0") \
  X(EV_MUL_OVERFLOW, ZKE_ASSERT, "mul_div_mod.py:64 (1-is_mul)*overflow == 0")              \
  /* PUSH: execution/push.py:6-33 */                                                        \
  X(EV_PUSH_LEN_UNSAT, ZKE_UNSAT, "push.py:9 bytecode_length lookup unsat")                 \
  X(EV_PUSH_LEN_AMBIG, ZKE_AMBIG, "push.py:9 bytecode_length lookup ambiguous")             \
  X(EV_PUSH_CMP_RANGE, ZKE_ASSERT, "push.py:11 compare(): operand exceeds 8 bytes (instruction.py:449-450)") \
  X(EV_PUSH_RW_UNSAT, ZKE_UNSAT, "push.py:14 stack_push unsat")                             \
  X(EV_PUSH_RW_AMBIG, ZKE_AMBIG, "push.py:14 stack_push ambiguous")                         \
  X(EV_PUSH_VALUE_BYTES, ZKE_VALUE, "push.py:15 to_le_bytes(): half >= 2^128 -> OverflowError") \
  ZK_EVM_PUSH_BYTE(X, 0)                                                              \
  ZK_EVM_PUSH_BYTE(X, 1)                                                              \
  ZK_EVM_PUSH_BYTE(X, 2)                                                              \
  ZK_EVM_PUSH_BYTE(X, 3)                                                              \
  ZK_EVM_PUSH_BYTE(X, 4)                                                              \
  ZK_EVM_PUSH_BYTE(X, 5)                                                              \
  ZK_EVM_PUSH_BYTE(X, 6)                                                              \
  ZK_EVM_PUSH_BYTE(X, 7)                                                              \
  ZK_EVM_PUSH_BYTE(X, 8)                                                              \
  ZK_EVM_PUSH_BYTE(X, 9)                                                              \
  ZK_EVM_PUSH_BYTE(X, 10)                                                              \
  ZK_EVM_PUSH_BYTE(X, 11)                                                              \
  ZK_EVM_PUSH_BYTE(X, 12)                                                              \
  ZK_EVM_PUSH_BYTE(X, 13)                                                              \
  ZK_EVM_PUSH_BYTE(X, 14)                                                              \
  ZK_EVM_PUSH_BYTE(X, 15)                                                              \
  ZK_EVM_PUSH_BYTE(X, 16)                                                              \
  ZK_EVM_PUSH_BYTE(X, 17)                                                              \
  ZK_EVM_PUSH_BYTE(X, 18)                                                              \
  ZK_EVM_PUSH_BYTE(X, 19)                                                              \
  ZK_EVM_PUSH_BYTE(X, 20)                                                              \
  ZK_EVM_PUSH_BYTE(X, 21)                                                              \
  ZK_EVM_PUSH_BYTE(X, 22)                                                              \
  ZK_EVM_PUSH_BYTE(X, 23)                                                              \
  ZK_EVM_PUSH_BYTE(X, 24)                                                              \
  ZK_EVM_PUSH_BYTE(X, 25)                                                              \
  ZK_EVM_PUSH_BYTE(X, 26)                                                              \
  ZK_EVM_PUSH_BYTE(X, 27)                                                              \
  ZK_EVM_PUSH_BYTE(X, 28)                                                              \
  ZK_EVM_PUSH_BYTE(X, 29)                                                              \
  ZK_EVM_PUSH_BYTE(X, 30)                                                              \
  ZK_EVM_PUSH_BYTE(X, 31)                                                              \
  /* POP: execution/pop.py:4-14 */                                                          \
  X(EV_POP_RW_UNSAT, ZKE_UNSAT, "pop.py:7 stack_pop unsat")                                 \
  X(EV_POP_RW_AMBIG, ZKE_AMBIG, "pop.py:7 stack_pop ambiguous")                             \
  /* SHA3: execution/sha3.py:6-55 */                                                        \
  X(EV_SHA_OFF_UNSAT, ZKE_UNSAT, "sha3.py:10 stack_pop offset unsat")                       \
  X(EV_SHA_OFF_AMBIG, ZKE_AMBIG, "sha3.py:10 stack_pop offset ambiguous")                   \
  X(EV_SHA_SIZE_UNSAT, ZKE_UNSAT, "sha3.py:12 stack_pop size unsat")                        \
  X(EV_SHA_SIZE_AMBIG, ZKE_AMBIG, "sha3.py:12 stack_pop size ambiguous")                    \
  X(EV_SHA_VAL_UNSAT, ZKE_UNSAT, "sha3.py:14 stack_push unsat")                             \
  X(EV_SHA_VAL_AMBIG, ZKE_AMBIG, "sha3.py:14 stack_push ambiguous")                         \
  X(EV_SHA_LEN_BYTES, ZKE_VALUE, "instruction.py:1123,481 to_le_bytes(size): half >= 2^128 -> OverflowError") \
  X(EV_SHA_LEN_RANGE, ZKE_RANGE, "instruction.py:1123,482-483 size does not fit 5 bytes")   \
  X(EV_SHA_OFF_BYTES, ZKE_VALUE, "instruction.py:1126,481 to_le_bytes(offset) -> OverflowError") \
  X(EV_SHA_OFF_RANGE, ZKE_RANGE, "instruction.py:1126,482-483 offset does not fit 5 bytes") \
  X(EV_SHA_COPY_UNSAT, ZKE_UNSAT, "sha3.py:20-30 copy_table lookup unsat")                  \
  X(EV_SHA_COPY_AMBIG, ZKE_AMBIG, "sha3.py:20-30 copy_table lookup ambiguous")              \
  X(EV_SHA_KECCAK_UNSAT, ZKE_UNSAT, "sha3.py:34 keccak_table lookup unsat")                 \
  X(EV_SHA_KECCAK_AMBIG, ZKE_AMBIG, "sha3.py:34 keccak_table lookup ambiguous")             \
  X(EV_SHA_HASH_EQ, ZKE_ASSERT, "sha3.py:35-38 keccak output == pushed word")               \
  X(EV_SHA_MEMSIZE_RANGE, ZKE_RANGE, "instruction.py:1164-1166 memory word size does not fit 4 bytes") \
  X(EV_SHA_MAX_RANGE, ZKE_ASSERT, "instruction.py:1167-1169,449-450 max(): operand exceeds 4 bytes") \
  X(EV_SHA_WORDSIZE_RANGE, ZKE_RANGE, "instruction.py:1189 copy word size does not fit 4 bytes") \
  X(EV_SHA_GASCOST_RANGE, ZKE_RANGE, "instruction.py:1191 copier gas cost does not fit 8 bytes") \
  /* CALLDATACOPY: execution/calldatacopy.py:6-62 */                                        \
  X(EV_CDC_MOFF_UNSAT, ZKE_UNSAT, "calldatacopy.py:9 stack_pop memory_offset unsat")        \
  X(EV_CDC_MOFF_AMBIG, ZKE_AMBIG, "calldatacopy.py:9 stack_pop memory_offset ambiguous")    \
  X(EV_CDC_DOFF_UNSAT, ZKE_UNSAT, "calldatacopy.py:10 stack_pop data_offset unsat")         \
  X(EV_CDC_DOFF_AMBIG, ZKE_AMBIG, "calldatacopy.py:10 stack_pop data_offset ambiguous")     \
  X(EV_CDC_LEN_UNSAT, ZKE_UNSAT, "calldatacopy.py:11 stack_pop length unsat")               \
  X(EV_CDC_LEN_AMBIG, ZKE_AMBIG, "calldatacopy.py:11 stack_pop length ambiguous")           \
  X(EV_CDC_LEN_BYTES, ZKE_VALUE, "calldatacopy.py:14 to_le_bytes(length) -> OverflowError") \
  X(EV_CDC_LEN_RANGE, ZKE_RANGE, "calldatacopy.py:14 length does not fit 5 bytes")          \
  X(EV_CDC_MOFF_BYTES, ZKE_VALUE, "calldatacopy.py:14 to_le_bytes(memory_offset) -> OverflowError") \
  X(EV_CDC_MOFF_RANGE, ZKE_RANGE, "calldatacopy.py:14 memory_offset does not fit 5 bytes")  \
  X(EV_CDC_DOFF_BYTES, ZKE_VALUE, "calldatacopy.py:15 to_le_bytes(data_offset) -> OverflowError") \
  X(EV_CDC_DOFF_RANGE, ZKE_RANGE, "calldatacopy.py:15 data_offset does not fit 5 bytes")    \
  X(EV_CDC_CC1_UNSAT, ZKE_UNSAT, "calldatacopy.py:18,24 call_context lookup (TxId | CallerId) unsat") \
  X(EV_CDC_CC1_AMBIG, ZKE_AMBIG, "calldatacopy.py:18,24 call_context lookup ambiguous")     \
  X(EV_CDC_CC1_TYPE, ZKE_ASSERT, "instruction.py:880 .value(): call-context value is a Word") \
  X(EV_CDC_CC2_UNSAT, ZKE_UNSAT, "calldatacopy.py:19,25 call_context lookup CallDataLength unsat") \
  X(EV_CDC_CC2_AMBIG, ZKE_AMBIG, "calldatacopy.py:19,25 call_context lookup ambiguous")     \
  X(EV_CDC_CC2_TYPE, ZKE_ASSERT, "instruction.py:880 .value(): call-context value is a Word") \
  X(EV_CDC_CC3_UNSAT, ZKE_UNSAT, "calldatacopy.py:28 call_context lookup CallDataOffset unsat") \
  X(EV_CDC_CC3_AMBIG, ZKE_AMBIG, "calldatacopy.py:28 call_context lookup ambiguous")        \
  X(EV_CDC_CC3_TYPE, ZKE_ASSERT, "instruction.py:880 .value(): call-context value is a Word") \
  X(EV_CDC_MEMSIZE_RANGE, ZKE_RANGE, "instruction.py:1164-1166 memory word size does not fit 4 bytes") \
  X(EV_CDC_MAX_RANGE, ZKE_ASSERT, "instruction.py:1167-1169 max(): operand exceeds 4 bytes") \
  X(EV_CDC_WORDSIZE_RANGE, ZKE_RANGE, "instruction.py:1189 copy word size does not fit 4 bytes") \
  X(EV_CDC_GASCOST_RANGE, ZKE_RANGE, "instruction.py:1191 copier gas cost does not fit 8 bytes") \
  X(EV_CDC_SELECT_BOOL, ZKE_ASSERT, "calldatacopy.py:37-39 select(): is_root is not boolean") \
  X(EV_CDC_COPY_UNSAT, ZKE_UNSAT, "calldatacopy.py:41-51 copy_table lookup unsat")          \
  X(EV_CDC_COPY_AMBIG, ZKE_AMBIG, "calldatacopy.py:41-51 copy_table lookup ambiguous")      \
  /* MEMORY (MLOAD / MSTORE / MSTORE8): execution/memory.py:7-44 */                          \
  X(EV_MEM_ADDR_UNSAT, ZKE_UNSAT, "memory.py:10 stack_pop address unsat")                   \
  X(EV_MEM_ADDR_AMBIG, ZKE_AMBIG, "memory.py:10 stack_pop address ambiguous")               \
  X(EV_MEM_ADDR_BYTES, ZKE_VALUE, "memory.py:10, instruction.py:481 to_le_bytes(address) -> OverflowError") \
  X(EV_MEM_ADDR_RANGE, ZKE_RANGE, "memory.py:10, instruction.py:482-483 address does not fit 20 bytes") \
  X(EV_MEM_VAL_UNSAT, ZKE_UNSAT, "memory.py:17 stack_push (MLOAD) / stack_pop value unsat") \
  X(EV_MEM_VAL_AMBIG, ZKE_AMBIG, "memory.py:17 value lookup ambiguous")                     \
  X(EV_MEM_VAL_BYTES, ZKE_VALUE, "memory.py:18 value.to_le_bytes() -> OverflowError")       \
  X(EV_MEM_MEMSIZE_RANGE, ZKE_RANGE, "instruction.py:1140-1142 memory size does not fit 4 bytes") \
  X(EV_MEM_MAX_RANGE, ZKE_ASSERT, "instruction.py:1147-1149,449-450 max(): memory_word_size exceeds 4 bytes") \
  X(EV_MEM_BYTE_UNSAT, ZKE_UNSAT, "memory.py:26,30-36 memory_lookup unsat")                 \
  X(EV_MEM_BYTE_AMBIG, ZKE_AMBIG, "memory.py:26,30-36 memory_lookup ambiguous")             \
  X(EV_MEM_BYTE_TYPE, ZKE_ASSERT, "instruction.py:934 .value(): memory value is a Word")    \
  /* MSIZE (msize.py), GAS (gas.py), ISZERO (iszero.py), CMP = LT/GT/EQ (comparator.py), JUMP (jump.py), \
   * JUMPI (jumpi.py) */                                                                     \
  X(EV_MSZ_WORD, ZKE_ASSERT, "msize.py:12 Word.from_lo(memory_word_size * 32): >= 2^128")    \
  X(EV_MSZ_PUSH_UNSAT, ZKE_UNSAT, "msize.py:12 stack_push unsat")                            \
  X(EV_MSZ_PUSH_AMBIG, ZKE_AMBIG, "msize.py:12 stack_push ambiguous")                        \
  X(EV_MSZ_EQ, ZKE_ASSERT, "msize.py:11-13 pushed word == memory_word_size * 32")            \
  X(EV_GAS_OPCODE, ZKE_ASSERT, "gas.py:9 opcode == GAS")                                     \
  X(EV_GAS_WORD, ZKE_ASSERT, "gas.py:12 Word.from_lo(gas_left - 2): >= 2^128")               \
  X(EV_GAS_PUSH_UNSAT, ZKE_UNSAT, "gas.py:13 stack_push unsat")                              \
  X(EV_GAS_PUSH_AMBIG, ZKE_AMBIG, "gas.py:13 stack_push ambiguous")                          \
  X(EV_GAS_EQ, ZKE_ASSERT, "gas.py:11-14 pushed word == gas_left - 2")                       \
  X(EV_ISZ_POP_UNSAT, ZKE_UNSAT, "iszero.py:8 stack_pop unsat")                              \
  X(EV_ISZ_POP_AMBIG, ZKE_AMBIG, "iszero.py:8 stack_pop ambiguous")                          \
  X(EV_ISZ_PUSH_UNSAT, ZKE_UNSAT, "iszero.py:12 stack_push unsat")                           \
  X(EV_ISZ_PUSH_AMBIG, ZKE_AMBIG, "iszero.py:12 stack_push ambiguous")                       \
  X(EV_ISZ_EQ, ZKE_ASSERT, "iszero.py:10-13 pushed word == is_zero_word(value)")             \
  X(EV_CMP_A_UNSAT, ZKE_UNSAT, "comparator.py:13 stack_pop a unsat")                         \
  X(EV_CMP_A_AMBIG, ZKE_AMBIG, "comparator.py:13 stack_pop a ambiguous")                     \
  X(EV_CMP_B_UNSAT, ZKE_UNSAT, "comparator.py:14 stack_pop b unsat")                         \
  X(EV_CMP_B_AMBIG, ZKE_AMBIG, "comparator.py:14 stack_pop b ambiguous")                     \
  X(EV_CMP_C_UNSAT, ZKE_UNSAT, "comparator.py:15 stack_push c unsat")                        \
  X(EV_CMP_C_AMBIG, ZKE_AMBIG, "comparator.py:15 stack_push c ambiguous")                    \
  X(EV_CMP_RANGE_LO, ZKE_ASSERT, "comparator.py:24, instruction.py:449-450 compare(lo halves): operand exceeds 16 bytes") \
  X(EV_CMP_RANGE_HI, ZKE_ASSERT, "comparator.py:27 compare(hi halves): operand exceeds 16 bytes") \
  X(EV_CMP_EQ, ZKE_ASSERT, "comparator.py:34-37 pushed word == result")                      \
  X(EV_JMP_OPCODE, ZKE_ASSERT, "jump.py:9 opcode == JUMP")                                   \
  X(EV_JMP_DEST_UNSAT, ZKE_UNSAT, "jump.py:13 stack_pop dest unsat")                         \
  X(EV_JMP_DEST_AMBIG, ZKE_AMBIG, "jump.py:13 stack_pop dest ambiguous")                     \
  X(EV_JMP_DEST_HI, ZKE_ASSERT, "jump.py:14 dest.hi == 0")                                   \
  X(EV_JMP_AT_UNSAT, ZKE_UNSAT, "jump.py:18 opcode_lookup_at(dest) unsat")                   \
  X(EV_JMP_AT_AMBIG, ZKE_AMBIG, "jump.py:18 opcode_lookup_at(dest) ambiguous")               \
  X(EV_JMP_NOT_JUMPDEST, ZKE_ASSERT, "jump.py:18 code at dest == JUMPDEST")                  \
  X(EV_JMPI_OPCODE, ZKE_ASSERT, "jumpi.py:9 opcode == JUMPI")                                \
  X(EV_JMPI_DEST_UNSAT, ZKE_UNSAT, "jumpi.py:13 stack_pop dest unsat")                       \
  X(EV_JMPI_DEST_AMBIG, ZKE_AMBIG, "jumpi.py:13 stack_pop dest ambiguous")                   \
  X(EV_JMPI_DEST_HI, ZKE_ASSERT, "jumpi.py:14 dest.hi == 0")                                 \
  X(EV_JMPI_COND_UNSAT, ZKE_UNSAT, "jumpi.py:17 stack_pop cond unsat")                       \
  X(EV_JMPI_COND_AMBIG, ZKE_AMBIG, "jumpi.py:17 stack_pop cond ambiguous")                   \
  /* CALLER / CALLVALUE / CALLDATASIZE / ADDRESS / RETURNDATASIZE (caller.py, callvalue.py,          \
   * calldatasize.py, address.py, returndatasize.py): one call-context read pushed on the stack; \
   * CODESIZE (codesize.py): the bytecode length pushed on the stack */                         \
  X(EV_CCP_OPCODE, ZKE_ASSERT, "caller.py:9 (and siblings) opcode == the gadget's opcode")    \
  X(EV_CCP_CC_UNSAT, ZKE_UNSAT, "caller.py:10 call_context_lookup unsat")                     \
  X(EV_CCP_CC_AMBIG, ZKE_AMBIG, "caller.py:10 call_context_lookup ambiguous")                 \
  X(EV_CCP_CC_TYPE, ZKE_ASSERT, "calldatasize.py:14, instruction.py:880 .value(): the call-context value is a Word") \
  X(EV_CCP_WORD, ZKE_ASSERT, "calldatasize.py:14 Word.from_lo(value): >= 2^128")              \
  X(EV_CCP_PUSH_UNSAT, ZKE_UNSAT, "caller.py:15 stack_push unsat")                            \
  X(EV_CCP_PUSH_AMBIG, ZKE_AMBIG, "caller.py:15 stack_push ambiguous")                        \
  X(EV_CCP_EQ, ZKE_ASSERT, "caller.py:13-16 pushed word == call-context value")               \
  X(EV_CSZ_OPCODE, ZKE_ASSERT, "codesize.py:9 opcode == CODESIZE")                            \
  X(EV_CSZ_LEN_UNSAT, ZKE_UNSAT, "codesize.py:10 bytecode_length lookup unsat")               \
  X(EV_CSZ_LEN_AMBIG, ZKE_AMBIG, "codesize.py:10 bytecode_length lookup ambiguous")           \
  X(EV_CSZ_WORD, ZKE_ASSERT, "codesize.py:11 Word.from_lo(code_size): >= 2^128")              \
  X(EV_CSZ_PUSH_UNSAT, ZKE_UNSAT, "codesize.py:11 stack_push unsat")                          \
  X(EV_CSZ_PUSH_AMBIG, ZKE_AMBIG, "codesize.py:11 stack_push ambiguous")                      \
  X(EV_CSZ_EQ, ZKE_ASSERT, "codesize.py:11 pushed word == code size")                         \
  /* BITWISE = AND / OR / XOR (bitwise.py), NOT (not_.py), BYTE (byte.py) */                     \
  X(EV_BW_A_UNSAT, ZKE_UNSAT, "bitwise.py:9 stack_pop a unsat")                               \
  X(EV_BW_A_AMBIG, ZKE_AMBIG, "bitwise.py:9 stack_pop a ambiguous")                           \
  X(EV_BW_B_UNSAT, ZKE_UNSAT, "bitwise.py:10 stack_pop b unsat")                              \
  X(EV_BW_B_AMBIG, ZKE_AMBIG, "bitwise.py:10 stack_pop b ambiguous")                          \
  X(EV_BW_C_UNSAT, ZKE_UNSAT, "bitwise.py:11 stack_push c unsat")                             \
  X(EV_BW_C_AMBIG, ZKE_AMBIG, "bitwise.py:11 stack_push c ambiguous")                         \
  X(EV_BW_BYTES, ZKE_VALUE, "bitwise.py:13-15 to_le_bytes(): half >= 2^128 -> OverflowError") \
  X(EV_BW_TAG, ZKE_VALUE, "bitwise.py:19 FixedTableTag(tag): not a valid tag -> ValueError")  \
  X(EV_BW_FIXED_UNSAT, ZKE_UNSAT, "bitwise.py:19 fixed_lookup(tag, a[i], b[i], c[i]) unsat")  \
  X(EV_BW_FIXED_AMBIG, ZKE_AMBIG, "bitwise.py:19 fixed_lookup ambiguous")                     \
  X(EV_NOT_A_UNSAT, ZKE_UNSAT, "not_.py:9 stack_pop unsat")                                   \
  X(EV_NOT_A_AMBIG, ZKE_AMBIG, "not_.py:9 stack_pop ambiguous")                               \
  X(EV_NOT_A_BYTES, ZKE_VALUE, "not_.py:10 a.to_le_bytes() -> OverflowError")                 \
  X(EV_NOT_B_UNSAT, ZKE_UNSAT, "not_.py:11 stack_push unsat")                                 \
  X(EV_NOT_B_AMBIG, ZKE_AMBIG, "not_.py:11 stack_push ambiguous")                             \
  X(EV_NOT_B_BYTES, ZKE_VALUE, "not_.py:12 b.to_le_bytes() -> OverflowError")                 \
  X(EV_NOT_FIXED_UNSAT, ZKE_UNSAT, "not_.py:17 fixed_lookup(BitwiseXor, a[i], b[i], 255) unsat") \
  X(EV_NOT_FIXED_AMBIG, ZKE_AMBIG, "not_.py:17 fixed_lookup ambiguous")                       \
  X(EV_BYTE_A_UNSAT, ZKE_UNSAT, "byte.py:9 stack_pop index unsat")                            \
  X(EV_BYTE_A_AMBIG, ZKE_AMBIG, "byte.py:9 stack_pop index ambiguous")                        \
  X(EV_BYTE_B_UNSAT, ZKE_UNSAT, "byte.py:10 stack_pop value unsat")                           \
  X(EV_BYTE_B_AMBIG, ZKE_AMBIG, "byte.py:10 stack_pop value ambiguous")                       \
  X(EV_BYTE_C_UNSAT, ZKE_UNSAT, "byte.py:11 stack_push unsat")                                \
  X(EV_BYTE_C_AMBIG, ZKE_AMBIG, "byte.py:11 stack_push ambiguous")                            \
  X(EV_BYTE_BYTES, ZKE_VALUE, "byte.py:13-14 to_le_bytes() -> OverflowError")                 \
  X(EV_BYTE_EQ, ZKE_ASSERT, "byte.py:30-33 pushed word == selected byte")                     \
  /* SCMP = SLT / SGT (slt_sgt.py), SIGNEXTEND (signextend.py) */                                \
  X(EV_SCMP_A_UNSAT, ZKE_UNSAT, "slt_sgt.py:12 stack_pop a unsat")                            \
  X(EV_SCMP_A_AMBIG, ZKE_AMBIG, "slt_sgt.py:12 stack_pop a ambiguous")                        \
  X(EV_SCMP_B_UNSAT, ZKE_UNSAT, "slt_sgt.py:13 stack_pop b unsat")                            \
  X(EV_SCMP_B_AMBIG, ZKE_AMBIG, "slt_sgt.py:13 stack_pop b ambiguous")                        \
  X(EV_SCMP_C_UNSAT, ZKE_UNSAT, "slt_sgt.py:14 stack_push c unsat")                           \
  X(EV_SCMP_C_AMBIG, ZKE_AMBIG, "slt_sgt.py:14 stack_push c ambiguous")                       \
  X(EV_SCMP_BYTES, ZKE_VALUE, "slt_sgt.py:21-23 to_le_bytes(): half >= 2^128 -> OverflowError") \
  X(EV_SCMP_C_MSB, ZKE_ASSERT, "slt_sgt.py:27 c8s[31] == 0")                                  \
  X(EV_SCMP_EQ, ZKE_ASSERT, "slt_sgt.py:36-44 result == signed a < b")                        \
  X(EV_SEXT_IDX_UNSAT, ZKE_UNSAT, "signextend.py:9 stack_pop index unsat")                    \
  X(EV_SEXT_IDX_AMBIG, ZKE_AMBIG, "signextend.py:9 stack_pop index ambiguous")                \
  X(EV_SEXT_VAL_UNSAT, ZKE_UNSAT, "signextend.py:10 stack_pop value unsat")                   \
  X(EV_SEXT_VAL_AMBIG, ZKE_AMBIG, "signextend.py:10 stack_pop value ambiguous")               \
  X(EV_SEXT_RES_UNSAT, ZKE_UNSAT, "signextend.py:11 stack_push result unsat")                 \
  X(EV_SEXT_RES_AMBIG, ZKE_AMBIG, "signextend.py:11 stack_push result ambiguous")             \
  X(EV_SEXT_BYTES, ZKE_VALUE, "signextend.py:13-15 to_le_bytes() -> OverflowError")           \
  X(EV_SEXT_SIGN_UNSAT, ZKE_UNSAT, "signextend.py:44 sign_byte_lookup(selected_byte, sign_byte) unsat") \
  X(EV_SEXT_SIGN_AMBIG, ZKE_AMBIG, "signextend.py:44 sign_byte_lookup ambiguous")             \
  /* BlockCtx = COINBASE / TIMESTAMP / NUMBER / PREVRANDAO / GASLIMIT / CHAINID / BASEFEE (block_ctx.py), \
   * ORIGIN (origin.py), GASPRICE (gasprice.py): a block-table or tx-table word pushed on the stack */ \
  X(EV_BLK_OPCODE, ZKE_VALUE, "block_ctx.py:10-24 opcode is none of the seven: `op` unbound -> UnboundLocalError") \
  X(EV_BLK_CTX_UNSAT, ZKE_UNSAT, "block_ctx.py:26 block_context_lookup_word unsat")           \
  X(EV_BLK_CTX_AMBIG, ZKE_AMBIG, "block_ctx.py:26 block_context_lookup_word ambiguous")       \
  X(EV_BLK_PUSH_UNSAT, ZKE_UNSAT, "block_ctx.py:27 stack_push unsat")                         \
  X(EV_BLK_PUSH_AMBIG, ZKE_AMBIG, "block_ctx.py:27 stack_push ambiguous")                     \
  X(EV_BLK_EQ, ZKE_ASSERT, "block_ctx.py:27 pushed word == block-context word")               \
  X(EV_TXC_TXID_UNSAT, ZKE_UNSAT, "origin.py:8 / gasprice.py:8 call_context_lookup(TxId) unsat") \
  X(EV_TXC_TXID_AMBIG, ZKE_AMBIG, "origin.py:8 call_context_lookup(TxId) ambiguous")          \
  X(EV_TXC_TXID_TYPE, ZKE_ASSERT, "instruction.py:880 .value(): TxId is a Word")              \
  X(EV_TXC_OPCODE, ZKE_ASSERT, "origin.py:10 / gasprice.py:10 opcode == ORIGIN / GASPRICE")   \
  X(EV_TXC_TX_UNSAT, ZKE_UNSAT, "origin.py:11 tx_context_lookup_word unsat")                  \
  X(EV_TXC_TX_AMBIG, ZKE_AMBIG, "origin.py:11 tx_context_lookup_word ambiguous")              \
  X(EV_TXC_PUSH_UNSAT, ZKE_UNSAT, "origin.py:15 stack_push unsat")                            \
  X(EV_TXC_PUSH_AMBIG, ZKE_AMBIG, "origin.py:15 stack_push ambiguous")                        \
  X(EV_TXC_EQ, ZKE_ASSERT, "origin.py:13-16 pushed word == tx-context word")                  \
  /* SHL_SHR (shl_shr.py): push == pop2 << pop1 / pop2 >> pop1 through a division witness */       \
  X(EV_SH_P1_UNSAT, ZKE_UNSAT, "shl_shr.py:10 stack_pop shift unsat")                         \
  X(EV_SH_P1_AMBIG, ZKE_AMBIG, "shl_shr.py:10 stack_pop shift ambiguous")                     \
  X(EV_SH_P2_UNSAT, ZKE_UNSAT, "shl_shr.py:11 stack_pop value unsat")                         \
  X(EV_SH_P2_AMBIG, ZKE_AMBIG, "shl_shr.py:11 stack_pop value ambiguous")                     \
  X(EV_SH_PUSH_UNSAT, ZKE_UNSAT, "shl_shr.py:12 stack_push unsat")                            \
  X(EV_SH_PUSH_AMBIG, ZKE_AMBIG, "shl_shr.py:12 stack_push ambiguous")                        \
  X(EV_SH_BYTES, ZKE_VALUE, "shl_shr.py:106 shift.to_le_bytes(): half >= 2^128 -> OverflowError") \
  X(EV_SH_REM_WORD, ZKE_ASSERT, "shl_shr.py:117 Word(dividend - quotient * divisor): >= 2^256") \
  X(EV_SH_REM_NEG, ZKE_VALUE, "shl_shr.py:117 Word(negative int): to_bytes -> OverflowError")  \
  X(EV_SH_SELECT, ZKE_ASSERT, "shl_shr.py:59-66 Word.select / +: a half >= 2^128 (arithmetic.py:110-114)") \
  X(EV_SH_POP2, ZKE_ASSERT, "shl_shr.py:59-62 pop2 == quotient*is_shl + dividend*is_shr")      \
  X(EV_SH_PUSH_EQ, ZKE_ASSERT, "shl_shr.py:63-65 push == dividend*is_shl + quotient*is_shr*(1 - divisor_is_zero)") \
  X(EV_SH_REM_LT, ZKE_ASSERT, "shl_shr.py:78-79 divisor != 0 => remainder < divisor")           \
  X(EV_SH_SHL_REM0, ZKE_ASSERT, "shl_shr.py:82-83 SHL => remainder == 0")                       \
  X(EV_SH_TO64, ZKE_VALUE, "instruction.py:604 to_64s(quotient): half >= 2^128 -> OverflowError") \
  X(EV_SH_CARRY_LO, ZKE_RANGE, "instruction.py:626 range_check(carry_lo, 9)")                   \
  X(EV_SH_CARRY_HI, ZKE_RANGE, "instruction.py:627 range_check(carry_hi, 9)")                   \
  X(EV_SH_OVERFLOW, ZKE_ASSERT, "shl_shr.py:87 is_shr * overflow == 0")                         \
  X(EV_SH_POW2_UNSAT, ZKE_UNSAT, "shl_shr.py:91 pow2_lookup(shf0, divisor) unsat")              \
  X(EV_SH_POW2_AMBIG, ZKE_AMBIG, "shl_shr.py:91 pow2_lookup ambiguous")                         \
  /* STOP: execution/stop.py:7-51 */                                                        \
  X(EV_STOP_LEN_UNSAT, ZKE_UNSAT, "stop.py:11 bytecode_length lookup unsat")                \
  X(EV_STOP_LEN_AMBIG, ZKE_AMBIG, "stop.py:11 bytecode_length lookup ambiguous")            \
  X(EV_STOP_CMP_RANGE, ZKE_ASSERT, "stop.py:12-14 compare(): operand exceeds 8 bytes")      \
  X(EV_STOP_OP_UNSAT, ZKE_UNSAT, "stop.py:18 opcode_lookup unsat")                          \
  X(EV_STOP_OP_AMBIG, ZKE_AMBIG, "stop.py:18 opcode_lookup ambiguous")                      \
  X(EV_STOP_RESP_OPCODE, ZKE_UNSAT, "stop.py:18 responsible_opcode_lookup")                 \
  X(EV_STOP_CC_UNSAT, ZKE_UNSAT, "stop.py:22 call_context IsSuccess lookup unsat")          \
  X(EV_STOP_CC_AMBIG, ZKE_AMBIG, "stop.py:22 call_context IsSuccess lookup ambiguous")      \
  X(EV_STOP_CC_TYPE, ZKE_ASSERT, "stop.py:22 .value(): IsSuccess is a Word")                \
  X(EV_STOP_IS_SUCCESS, ZKE_ASSERT, "stop.py:23 is_success == 1")                           \
  X(EV_STOP_ROOT_ENDTX, ZKE_ASSERT, "stop.py:26-27 is_root == (next state is EndTx)")       \
  X(EV_STOP_RWC, ZKE_ASSERT, "stop.py:31-34 root: rw_counter + 1")                          \
  X(EV_STOP_CALL_ID, ZKE_ASSERT, "stop.py:31-34 root: call_id same")                        \
  /* step_state_transition_to_restored_context, instruction.py:293-363: lookup 0 = CallerId,  \
   * 1..8 = caller IsRoot, IsCreate, CodeHash, ProgramCounter, StackPointer, GasLeft,          \
   * MemorySize, ReversibleWriteCounter, 9..11 = writes LastCalleeId / ReturnDataOffset / Length */ \
  ZK_EVM_RESTORE_LOOKUP(X, 0)                                                          \
  ZK_EVM_RESTORE_LOOKUP(X, 1)                                                          \
  ZK_EVM_RESTORE_LOOKUP(X, 2)                                                          \
  ZK_EVM_RESTORE_LOOKUP(X, 3)                                                          \
  ZK_EVM_RESTORE_LOOKUP(X, 4)                                                          \
  ZK_EVM_RESTORE_LOOKUP(X, 5)                                                          \
  ZK_EVM_RESTORE_LOOKUP(X, 6)                                                          \
  ZK_EVM_RESTORE_LOOKUP(X, 7)                                                          \
  ZK_EVM_RESTORE_LOOKUP(X, 8)                                                          \
  ZK_EVM_RESTORE_LOOKUP(X, 9)                                                          \
  ZK_EVM_RESTORE_LOOKUP(X, 10)                                                          \
  ZK_EVM_RESTORE_LOOKUP(X, 11)                                                          \
  X(EV_RST_VALUE_TYPE, ZKE_ASSERT, "instruction.py:349-361 .value(): a restored field is a Word") \
  X(EV_RST_RWC, ZKE_ASSERT, "instruction.py:348 rw_counter + delta")                        \
  X(EV_RST_CALL_ID, ZKE_ASSERT, "instruction.py:349 call_id -> caller_id")                  \
  X(EV_RST_IS_ROOT, ZKE_ASSERT, "instruction.py:350 is_root -> caller's")                   \
  X(EV_RST_IS_CREATE, ZKE_ASSERT, "instruction.py:351 is_create -> caller's")               \
  X(EV_RST_CODE_HASH, ZKE_ASSERT, "instruction.py:352 code_hash -> caller's")               \
  X(EV_RST_PC, ZKE_ASSERT, "instruction.py:353 program_counter -> caller's")                \
  X(EV_RST_SP, ZKE_ASSERT, "instruction.py:354 stack_pointer -> caller's")                  \
  X(EV_RST_GAS, ZKE_ASSERT, "instruction.py:356 gas_left -> caller's + returned")           \
  X(EV_RST_MEM, ZKE_ASSERT, "instruction.py:357 memory_word_size -> caller's")              \
  X(EV_RST_REV, ZKE_ASSERT, "instruction.py:359-361 reversible_write_counter -> caller's + own") \
  /* shared epilogue: step_state_transition_in_same_context, instruction.py:365-394 */      \
  X(EV_SC_RESP_OPCODE, ZKE_UNSAT, "instruction.py:376,779-782 ResponsibleOpcode fixed lookup") \
  X(EV_SC_OPCODE_VALUE, ZKE_VALUE, "instruction.py:378 Opcode(opcode.n): not a valid opcode -> ValueError") \
  X(EV_SC_GAS_RANGE, ZKE_RANGE, "instruction.py:379,529-534 gas_left - gas_cost fits 8 bytes") \
  X(EV_SC_RWC, ZKE_ASSERT, "instruction.py:381-394 rw_counter transition")                  \
  X(EV_SC_PC, ZKE_ASSERT, "instruction.py:381-394 program_counter transition")              \
  X(EV_SC_SP, ZKE_ASSERT, "instruction.py:381-394 stack_pointer transition")                \
  X(EV_SC_GAS, ZKE_ASSERT, "instruction.py:381-394 gas_left transition")                    \
  X(EV_SC_MEM, ZKE_ASSERT, "instruction.py:381-394 memory_word_size transition")            \
  X(EV_SC_REV, ZKE_ASSERT, "instruction.py:381-394 reversible_write_counter transition")    \
  X(EV_SC_LOG, ZKE_ASSERT, "instruction.py:381-394 log_id transition")                      \
  X(EV_SC_CALL_ID, ZKE_ASSERT, "instruction.py:381-394 call_id same")                       \
  X(EV_SC_IS_ROOT, ZKE_ASSERT, "instruction.py:381-394 is_root same")                       \
  X(EV_SC_IS_CREATE, ZKE_ASSERT, "instruction.py:381-394 is_create same")                   \
  X(EV_SC_CODE_HASH, ZKE_ASSERT, "instruction.py:381-394 code_hash same") \
  X(EV_ETX_CC_TXID_UNSAT, ZKE_UNSAT, "end_tx.py:8 call_context_lookup(TxId) unsat") \
  X(EV_ETX_CC_TXID_AMBIG, ZKE_AMBIG, "end_tx.py:8 call_context_lookup(TxId) ambiguous") \
  X(EV_ETX_CC_TXID_TYPE, ZKE_ASSERT, "end_tx.py:8 call_context_lookup(TxId): .value() of a Word-typed cell (arithmetic.py:186-189)") \
  X(EV_ETX_CC_PERSIST_UNSAT, ZKE_UNSAT, "end_tx.py:9 call_context_lookup(IsPersistent) unsat") \
  X(EV_ETX_CC_PERSIST_AMBIG, ZKE_AMBIG, "end_tx.py:9 call_context_lookup(IsPersistent) ambiguous") \
  X(EV_ETX_CC_PERSIST_TYPE, ZKE_ASSERT, "end_tx.py:9 call_context_lookup(IsPersistent): .value() of a Word-typed cell (arithmetic.py:186-189)") \
  X(EV_ETX_TX_INVALID_UNSAT, ZKE_UNSAT, "end_tx.py:10 tx_context_lookup(TxInvalid) unsat") \
  X(EV_ETX_TX_INVALID_AMBIG, ZKE_AMBIG, "end_tx.py:10 tx_context_lookup(TxInvalid) ambiguous") \
  X(EV_ETX_TX_INVALID_TYPE, ZKE_ASSERT, "end_tx.py:10 tx_context_lookup(TxInvalid): .value() of a Word-typed cell (arithmetic.py:186-189)") \
  X(EV_ETX_TX_GAS_UNSAT, ZKE_UNSAT, "end_tx.py:13 tx_context_lookup(Gas) unsat") \
  X(EV_ETX_TX_GAS_AMBIG, ZKE_AMBIG, "end_tx.py:13 tx_context_lookup(Gas) ambiguous") \
  X(EV_ETX_TX_GAS_TYPE, ZKE_ASSERT, "end_tx.py:13 tx_context_lookup(Gas): .value() of a Word-typed cell (arithmetic.py:186-189)") \
  X(EV_ETX_MAXREFUND_RANGE, ZKE_RANGE, "end_tx.py:15-17 constant_divmod(gas_used, 5, 8): range_check(quotient, 8)") \
  X(EV_ETX_REFUND_UNSAT, ZKE_UNSAT, "end_tx.py:18 tx_refund_read(tx_id) unsat") \
  X(EV_ETX_REFUND_AMBIG, ZKE_AMBIG, "end_tx.py:18 tx_refund_read(tx_id) ambiguous") \
  X(EV_ETX_REFUND_TYPE, ZKE_ASSERT, "end_tx.py:18 tx_refund_read(tx_id): .value() of a Word-typed cell (arithmetic.py:186-189)") \
  X(EV_ETX_MIN_RANGE, ZKE_ASSERT, "end_tx.py:19 min(max_refund, refund, 8): compare() operands < 256^8 (instruction.py:449-450)") \
  X(EV_ETX_INVALID_REFUND0, ZKE_ASSERT, "end_tx.py:22-23 tx invalid => effective_refund == 0") \
  X(EV_ETX_TX_GASPRICE_UNSAT, ZKE_UNSAT, "end_tx.py:26 tx_gas_price(tx_id) unsat") \
  X(EV_ETX_TX_GASPRICE_AMBIG, ZKE_AMBIG, "end_tx.py:26 tx_gas_price(tx_id) ambiguous") \
  X(EV_ETX_MUL1_OVERFLOW, ZKE_ASSERT, "end_tx.py:27 mul_word_by_u64: quotient_hi == 0 (instruction.py:595)") \
  X(EV_ETX_TX_CALLER_UNSAT, ZKE_UNSAT, "end_tx.py:28-30 tx_context_lookup_word(CallerAddress) unsat") \
  X(EV_ETX_TX_CALLER_AMBIG, ZKE_AMBIG, "end_tx.py:28-30 tx_context_lookup_word(CallerAddress) ambiguous") \
  X(EV_ETX_CALLER_BYTES, ZKE_VALUE, "end_tx.py:31 word_to_address: to_le_bytes of a half >= 2^128 -> OverflowError") \
  X(EV_ETX_CALLER_RANGE, ZKE_RANGE, "end_tx.py:31 word_to_address: bytes 20.. not zero (instruction.py:482-483)") \
  X(EV_ETX_BAL_CALLER_UNSAT, ZKE_UNSAT, "end_tx.py:32 add_balance(caller): account_write_word(Balance) unsat") \
  X(EV_ETX_BAL_CALLER_AMBIG, ZKE_AMBIG, "end_tx.py:32 add_balance(caller): account_write_word(Balance) ambiguous") \
  X(EV_ETX_BAL1_EQ, ZKE_ASSERT, "end_tx.py:32 add_balance: balance == balance_prev + value (instruction.py:997)") \
  X(EV_ETX_BAL1_CARRY, ZKE_ASSERT, "end_tx.py:32 add_balance: carry == 0 (instruction.py:998)") \
  X(EV_ETX_BLK_BASEFEE_UNSAT, ZKE_UNSAT, "end_tx.py:35 block_context_lookup_word(BaseFee) unsat") \
  X(EV_ETX_BLK_BASEFEE_AMBIG, ZKE_AMBIG, "end_tx.py:35 block_context_lookup_word(BaseFee) ambiguous") \
  X(EV_ETX_SUBWORD_RANGE, ZKE_ASSERT, "end_tx.py:36 sub_word: Word((diff_lo, diff_hi)) halves < 2^128 (arithmetic.py:110-114)") \
  X(EV_ETX_MUL2_OVERFLOW, ZKE_ASSERT, "end_tx.py:37 mul_word_by_u64(effective_tip, gas_used): quotient_hi == 0") \
  X(EV_ETX_BLK_COINBASE_UNSAT, ZKE_UNSAT, "end_tx.py:38 block_context_lookup_word(Coinbase) unsat") \
  X(EV_ETX_BLK_COINBASE_AMBIG, ZKE_AMBIG, "end_tx.py:38 block_context_lookup_word(Coinbase) ambiguous") \
  X(EV_ETX_COINBASE_BYTES, ZKE_VALUE, "end_tx.py:39 word_to_address(coinbase): OverflowError") \
  X(EV_ETX_COINBASE_RANGE, ZKE_RANGE, "end_tx.py:39 word_to_address(coinbase): bytes 20.. not zero") \
  X(EV_ETX_BAL_COINBASE_UNSAT, ZKE_UNSAT, "end_tx.py:40 add_balance(coinbase) unsat") \
  X(EV_ETX_BAL_COINBASE_AMBIG, ZKE_AMBIG, "end_tx.py:40 add_balance(coinbase) ambiguous") \
  X(EV_ETX_BAL2_EQ, ZKE_ASSERT, "end_tx.py:40 add_balance(coinbase): balance == balance_prev + reward") \
  X(EV_ETX_BAL2_CARRY, ZKE_ASSERT, "end_tx.py:40 add_balance(coinbase): carry == 0") \
  X(EV_ETX_RCPT_STATUS_UNSAT, ZKE_UNSAT, "end_tx.py:45 tx_receipt_write(PostStateOrStatus) unsat") \
  X(EV_ETX_RCPT_STATUS_AMBIG, ZKE_AMBIG, "end_tx.py:45 tx_receipt_write(PostStateOrStatus) ambiguous") \
  X(EV_ETX_RCPT_STATUS_TYPE, ZKE_ASSERT, "end_tx.py:45 tx_receipt_write(PostStateOrStatus): .value() of a Word-typed cell (arithmetic.py:186-189)") \
  X(EV_ETX_STATUS, ZKE_ASSERT, "end_tx.py:43-46 (1 - is_tx_invalid) * is_persistent == PostStateOrStatus") \
  X(EV_ETX_RCPT_LOG_UNSAT, ZKE_UNSAT, "end_tx.py:49 tx_receipt_write(LogLength) unsat") \
  X(EV_ETX_RCPT_LOG_AMBIG, ZKE_AMBIG, "end_tx.py:49 tx_receipt_write(LogLength) ambiguous") \
  X(EV_ETX_RCPT_LOG_TYPE, ZKE_ASSERT, "end_tx.py:49 tx_receipt_write(LogLength): .value() of a Word-typed cell (arithmetic.py:186-189)") \
  X(EV_ETX_LOGID, ZKE_ASSERT, "end_tx.py:50 log_id == curr.log_id") \
  X(EV_ETX_LOGID0, ZKE_ASSERT, "end_tx.py:52-53 tx invalid => log_id == 0") \
  X(EV_ETX_RCPT_PREVCUM_UNSAT, ZKE_UNSAT, "end_tx.py:60-62 tx_receipt_read(tx_id - 1, CumulativeGasUsed) unsat") \
  X(EV_ETX_RCPT_PREVCUM_AMBIG, ZKE_AMBIG, "end_tx.py:60-62 tx_receipt_read(tx_id - 1, CumulativeGasUsed) ambiguous") \
  X(EV_ETX_RCPT_PREVCUM_TYPE, ZKE_ASSERT, "end_tx.py:60-62 tx_receipt_read(tx_id - 1, CumulativeGasUsed): .value() of a Word-typed cell (arithmetic.py:186-189)") \
  X(EV_ETX_RCPT_CUM_UNSAT, ZKE_UNSAT, "end_tx.py:66 tx_receipt_write(CumulativeGasUsed) unsat") \
  X(EV_ETX_RCPT_CUM_AMBIG, ZKE_AMBIG, "end_tx.py:66 tx_receipt_write(CumulativeGasUsed) ambiguous") \
  X(EV_ETX_RCPT_CUM_TYPE, ZKE_ASSERT, "end_tx.py:66 tx_receipt_write(CumulativeGasUsed): .value() of a Word-typed cell (arithmetic.py:186-189)") \
  X(EV_ETX_CUMGAS, ZKE_ASSERT, "end_tx.py:64-67 previous cumulative gas + gas_used == CumulativeGasUsed") \
  X(EV_ETX_CC_NEXT_TXID_UNSAT, ZKE_UNSAT, "end_tx.py:73-75 call_context_lookup(TxId, call_id=next.rw_counter) unsat") \
  X(EV_ETX_CC_NEXT_TXID_AMBIG, ZKE_AMBIG, "end_tx.py:73-75 call_context_lookup(TxId, call_id=next.rw_counter) ambiguous") \
  X(EV_ETX_CC_NEXT_TXID_TYPE, ZKE_ASSERT, "end_tx.py:73-75 call_context_lookup(TxId, call_id=next.rw_counter): .value() of a Word-typed cell (arithmetic.py:186-189)") \
  X(EV_ETX_NEXT_TXID, ZKE_ASSERT, "end_tx.py:72-77 next tx id == tx_id + 1") \
  X(EV_ETX_RWC_BEGINTX, ZKE_ASSERT, "end_tx.py:79 rw_counter delta 10 - is_first_tx") \
  X(EV_ETX_RWC_ENDBLOCK, ZKE_ASSERT, "end_tx.py:84-86 rw_counter delta 9 - is_first_tx") \
  X(EV_ETX_CALLID_ENDBLOCK, ZKE_ASSERT, "end_tx.py:84-86 call_id same") \
  X(EV_EB_TXINVALID_TYPE, ZKE_ASSERT, "end_block.py:87-92 tx_row.value.value() of a Word-typed TxInvalid row") \
  X(EV_EB_EMPTY_VALID_TXS, ZKE_ASSERT, "end_block.py:118 empty block: total_valid_txs == 0") \
  X(EV_EB_EMPTY_WDS, ZKE_ASSERT, "end_block.py:119 empty block: total_withdrawals == 0") \
  X(EV_EB_CC_TXID_UNSAT, ZKE_UNSAT, "end_block.py:123 call_context_lookup(TxId) unsat") \
  X(EV_EB_CC_TXID_AMBIG, ZKE_AMBIG, "end_block.py:123 call_context_lookup(TxId) ambiguous") \
  X(EV_EB_CC_TXID_TYPE, ZKE_ASSERT, "end_block.py:123 call_context_lookup(TxId): .value() of a Word-typed cell (arithmetic.py:186-189)") \
  X(EV_EB_TXID_EQ, ZKE_ASSERT, "end_block.py:122-124 last tx id == total_txs") \
  X(EV_EB_BLK_GASLIMIT_UNSAT, ZKE_UNSAT, "end_block.py:127 block_context_lookup(GasLimit) unsat") \
  X(EV_EB_BLK_GASLIMIT_AMBIG, ZKE_AMBIG, "end_block.py:127 block_context_lookup(GasLimit) ambiguous") \
  X(EV_EB_BLK_GASLIMIT_TYPE, ZKE_ASSERT, "end_block.py:127 block_context_lookup(GasLimit): .value() of a Word-typed cell (arithmetic.py:186-189)") \
  X(EV_EB_RCPT_CUM_UNSAT, ZKE_UNSAT, "end_block.py:128-131 tx_receipt_read(total_txs, CumulativeGasUsed) unsat") \
  X(EV_EB_RCPT_CUM_AMBIG, ZKE_AMBIG, "end_block.py:128-131 tx_receipt_read(total_txs, CumulativeGasUsed) ambiguous") \
  X(EV_EB_RCPT_CUM_TYPE, ZKE_ASSERT, "end_block.py:128-131 tx_receipt_read(total_txs, CumulativeGasUsed): .value() of a Word-typed cell (arithmetic.py:186-189)") \
  X(EV_EB_GAS_CMP_RANGE, ZKE_ASSERT, "end_block.py:132 compare(gas_limit, cumulative_gas, 8): operands < 256^8") \
  X(EV_EB_GAS_LIMIT, ZKE_ASSERT, "end_block.py:133 cumulative gas <= gas limit") \
  X(EV_EB_WD_WORD, ZKE_ASSERT, "end_block.py:142 Word(amount * 1e9) >= 2^256 (arithmetic.py:117)") \
  X(EV_EB_WD_BAL_UNSAT, ZKE_UNSAT, "end_block.py:142 add_balance(withdrawal address) unsat") \
  X(EV_EB_WD_BAL_AMBIG, ZKE_AMBIG, "end_block.py:142 add_balance(withdrawal address) ambiguous") \
  X(EV_EB_WD_BAL_EQ, ZKE_ASSERT, "end_block.py:142 add_balance: balance == balance_prev + amount * 1e9") \
  X(EV_EB_WD_BAL_CARRY, ZKE_ASSERT, "end_block.py:142 add_balance: carry == 0") \
  X(EV_EB_TX_PAD_UNSAT, ZKE_UNSAT, "end_block.py:157-159 tx_context_lookup_word(total_txs + 1, CallerAddress) unsat") \
  X(EV_EB_TX_PAD_AMBIG, ZKE_AMBIG, "end_block.py:157-159 tx_context_lookup_word(total_txs + 1, CallerAddress) ambiguous") \
  X(EV_EB_TX_PAD_ZERO, ZKE_ASSERT, "end_block.py:156-161 the tx after the last one is padding (CallerAddress == 0)") \
  X(EV_EB_START1_UNSAT, ZKE_UNSAT, "end_block.py:170 rw_table_start_lookup(1) unsat") \
  X(EV_EB_START1_AMBIG, ZKE_AMBIG, "end_block.py:170 rw_table_start_lookup(1) ambiguous") \
  X(EV_EB_START2_UNSAT, ZKE_UNSAT, "end_block.py:171 rw_table_start_lookup(max_rws - total_rws - total_withdrawals) unsat") \
  X(EV_EB_START2_AMBIG, ZKE_AMBIG, "end_block.py:171 rw_table_start_lookup(max_rws - total_rws - total_withdrawals) ambiguous") \
  X(EV_EB_RWC_SAME, ZKE_ASSERT, "end_block.py:180-183 rw_counter same") \
  X(EV_EB_CALLID_SAME, ZKE_ASSERT, "end_block.py:180-183 call_id same") \
  X(EV_BT_CC_TXID_UNSAT, ZKE_UNSAT, "begin_tx.py:26 call_context_lookup(TxId, call_id) unsat") \
  X(EV_BT_CC_TXID_AMBIG, ZKE_AMBIG, "begin_tx.py:26 call_context_lookup(TxId, call_id) ambiguous") \
  X(EV_BT_CC_TXID_TYPE, ZKE_ASSERT, "begin_tx.py:26 call_context_lookup(TxId, call_id): .value() of a Word-typed cell (arithmetic.py:186-189)") \
  X(EV_BT_CC_REVEND_UNSAT, ZKE_UNSAT, "begin_tx.py:27 reversion_info: RwCounterEndOfReversion unsat") \
  X(EV_BT_CC_REVEND_AMBIG, ZKE_AMBIG, "begin_tx.py:27 reversion_info: RwCounterEndOfReversion ambiguous") \
  X(EV_BT_CC_REVEND_TYPE, ZKE_ASSERT, "begin_tx.py:27 reversion_info: RwCounterEndOfReversion: .value() of a Word-typed cell (arithmetic.py:186-189)") \
  X(EV_BT_CC_PERSIST_UNSAT, ZKE_UNSAT, "begin_tx.py:27 reversion_info: IsPersistent unsat") \
  X(EV_BT_CC_PERSIST_AMBIG, ZKE_AMBIG, "begin_tx.py:27 reversion_info: IsPersistent ambiguous") \
  X(EV_BT_CC_PERSIST_TYPE, ZKE_ASSERT, "begin_tx.py:27 reversion_info: IsPersistent: .value() of a Word-typed cell (arithmetic.py:186-189)") \
  X(EV_BT_CC_SUCCESS_UNSAT, ZKE_UNSAT, "begin_tx.py:29 call_context_lookup(IsSuccess) unsat") \
  X(EV_BT_CC_SUCCESS_AMBIG, ZKE_AMBIG, "begin_tx.py:29 call_context_lookup(IsSuccess) ambiguous") \
  X(EV_BT_CC_SUCCESS_TYPE, ZKE_ASSERT, "begin_tx.py:29 call_context_lookup(IsSuccess): .value() of a Word-typed cell (arithmetic.py:186-189)") \
  X(EV_BT_SUCCESS_EQ, ZKE_ASSERT, "begin_tx.py:28-31 IsSuccess == is_persistent") \
  X(EV_BT_FIRST_TXID, ZKE_ASSERT, "begin_tx.py:33-34 first step: tx_id == 1") \
  X(EV_BT_BLK_COINBASE_UNSAT, ZKE_UNSAT, "begin_tx.py:37 block_context_lookup_word(Coinbase) unsat") \
  X(EV_BT_BLK_COINBASE_AMBIG, ZKE_AMBIG, "begin_tx.py:37 block_context_lookup_word(Coinbase) ambiguous") \
  X(EV_BT_COINBASE_BYTES, ZKE_VALUE, "begin_tx.py:38 word_to_address: OverflowError") \
  X(EV_BT_COINBASE_RANGE, ZKE_RANGE, "begin_tx.py:38 word_to_address: bytes 20.. not zero") \
  X(EV_BT_TX_CALLER_UNSAT, ZKE_UNSAT, "begin_tx.py:40-42 tx_context_lookup_word(CallerAddress) unsat") \
  X(EV_BT_TX_CALLER_AMBIG, ZKE_AMBIG, "begin_tx.py:40-42 tx_context_lookup_word(CallerAddress) ambiguous") \
  X(EV_BT_CALLER_BYTES, ZKE_VALUE, "begin_tx.py:43 word_to_address: OverflowError") \
  X(EV_BT_CALLER_RANGE, ZKE_RANGE, "begin_tx.py:43 word_to_address: bytes 20.. not zero") \
  X(EV_BT_TX_CALLEE_UNSAT, ZKE_UNSAT, "begin_tx.py:44-46 tx_context_lookup_word(CalleeAddress) unsat") \
  X(EV_BT_TX_CALLEE_AMBIG, ZKE_AMBIG, "begin_tx.py:44-46 tx_context_lookup_word(CalleeAddress) ambiguous") \
  X(EV_BT_CALLEE_BYTES, ZKE_VALUE, "begin_tx.py:47 word_to_address: OverflowError") \
  X(EV_BT_CALLEE_RANGE, ZKE_RANGE, "begin_tx.py:47 word_to_address: bytes 20.. not zero") \
  X(EV_BT_TX_ISCREATE_UNSAT, ZKE_UNSAT, "begin_tx.py:48 tx_context_lookup(IsCreate) unsat") \
  X(EV_BT_TX_ISCREATE_AMBIG, ZKE_AMBIG, "begin_tx.py:48 tx_context_lookup(IsCreate) ambiguous") \
  X(EV_BT_TX_ISCREATE_TYPE, ZKE_ASSERT, "begin_tx.py:48 tx_context_lookup(IsCreate): .value() of a Word-typed cell (arithmetic.py:186-189)") \
  X(EV_BT_TX_VALUE_UNSAT, ZKE_UNSAT, "begin_tx.py:49 tx_context_lookup_word(Value) unsat") \
  X(EV_BT_TX_VALUE_AMBIG, ZKE_AMBIG, "begin_tx.py:49 tx_context_lookup_word(Value) ambiguous") \
  X(EV_BT_TX_CDLEN_UNSAT, ZKE_UNSAT, "begin_tx.py:50 tx_context_lookup(CallDataLength) unsat") \
  X(EV_BT_TX_CDLEN_AMBIG, ZKE_AMBIG, "begin_tx.py:50 tx_context_lookup(CallDataLength) ambiguous") \
  X(EV_BT_TX_CDLEN_TYPE, ZKE_ASSERT, "begin_tx.py:50 tx_context_lookup(CallDataLength): .value() of a Word-typed cell (arithmetic.py:186-189)") \
  X(EV_BT_CALLER_NONZERO, ZKE_ASSERT, "begin_tx.py:53 CallerAddress != 0") \
  X(EV_BT_TX_INVALID_UNSAT, ZKE_UNSAT, "begin_tx.py:63 tx_context_lookup(TxInvalid) unsat") \
  X(EV_BT_TX_INVALID_AMBIG, ZKE_AMBIG, "begin_tx.py:63 tx_context_lookup(TxInvalid) ambiguous") \
  X(EV_BT_TX_INVALID_TYPE, ZKE_ASSERT, "begin_tx.py:63 tx_context_lookup(TxInvalid): .value() of a Word-typed cell (arithmetic.py:186-189)") \
  X(EV_BT_TX_NONCE_UNSAT, ZKE_UNSAT, "begin_tx.py:64 tx_context_lookup(Nonce) unsat") \
  X(EV_BT_TX_NONCE_AMBIG, ZKE_AMBIG, "begin_tx.py:64 tx_context_lookup(Nonce) ambiguous") \
  X(EV_BT_TX_NONCE_TYPE, ZKE_ASSERT, "begin_tx.py:64 tx_context_lookup(Nonce): .value() of a Word-typed cell (arithmetic.py:186-189)") \
  X(EV_BT_ACC_NONCE_UNSAT, ZKE_UNSAT, "begin_tx.py:65 account_write(caller, Nonce) unsat") \
  X(EV_BT_ACC_NONCE_AMBIG, ZKE_AMBIG, "begin_tx.py:65 account_write(caller, Nonce) ambiguous") \
  X(EV_BT_ACC_NONCE_TYPE, ZKE_ASSERT, "begin_tx.py:65 account_write(caller, Nonce): .value() of a Word-typed cell (arithmetic.py:186-189)") \
  X(EV_BT_ACC_NONCE_PREV_TYPE, ZKE_ASSERT, "begin_tx.py:65 account_write: value_prev.value() of a Word-typed cell") \
  X(EV_BT_NONCE_EQ, ZKE_ASSERT, "begin_tx.py:68 nonce == nonce_prev + 1 - is_tx_invalid") \
  X(EV_BT_TX_GAS_UNSAT, ZKE_UNSAT, "begin_tx.py:72 tx_context_lookup(Gas) unsat") \
  X(EV_BT_TX_GAS_AMBIG, ZKE_AMBIG, "begin_tx.py:72 tx_context_lookup(Gas) ambiguous") \
  X(EV_BT_TX_GAS_TYPE, ZKE_ASSERT, "begin_tx.py:72 tx_context_lookup(Gas): .value() of a Word-typed cell (arithmetic.py:186-189)") \
  X(EV_BT_TX_GASPRICE_UNSAT, ZKE_UNSAT, "begin_tx.py:73 tx_gas_price unsat") \
  X(EV_BT_TX_GASPRICE_AMBIG, ZKE_AMBIG, "begin_tx.py:73 tx_gas_price ambiguous") \
  X(EV_BT_GASFEE_OVERFLOW, ZKE_ASSERT, "begin_tx.py:74 mul_word_by_u64(gas_price, gas): quotient_hi == 0") \
  X(EV_BT_TX_CDGAS_UNSAT, ZKE_UNSAT, "begin_tx.py:82 tx_context_lookup(CallDataGasCost) unsat") \
  X(EV_BT_TX_CDGAS_AMBIG, ZKE_AMBIG, "begin_tx.py:82 tx_context_lookup(CallDataGasCost) ambiguous") \
  X(EV_BT_TX_CDGAS_TYPE, ZKE_ASSERT, "begin_tx.py:82 tx_context_lookup(CallDataGasCost): .value() of a Word-typed cell (arithmetic.py:186-189)") \
  X(EV_BT_INITCODE_RANGE, ZKE_RANGE, "begin_tx.py:85-87 constant_divmod(len + 31, 32, 8): range_check") \
  X(EV_BT_TX_ALGAS_UNSAT, ZKE_UNSAT, "begin_tx.py:91 tx_context_lookup(AccessListGasCost) unsat") \
  X(EV_BT_TX_ALGAS_AMBIG, ZKE_AMBIG, "begin_tx.py:91 tx_context_lookup(AccessListGasCost) ambiguous") \
  X(EV_BT_TX_ALGAS_TYPE, ZKE_ASSERT, "begin_tx.py:91 tx_context_lookup(AccessListGasCost): .value() of a Word-typed cell (arithmetic.py:186-189)") \
  X(EV_BT_GAS_CMP_RANGE, ZKE_ASSERT, "begin_tx.py:96 compare(tx_gas, intrinsic, 31): operands < 256^31") \
  X(EV_BT_AL_COINBASE_UNSAT, ZKE_UNSAT, "begin_tx.py:106-108 add_account_to_access_list(coinbase) unsat") \
  X(EV_BT_AL_COINBASE_AMBIG, ZKE_AMBIG, "begin_tx.py:106-108 add_account_to_access_list(coinbase) ambiguous") \
  X(EV_BT_AL_COINBASE_TYPE, ZKE_ASSERT, "begin_tx.py:106-108 access list (coinbase): value_prev.value() of a Word-typed cell") \
  X(EV_BT_AL_COINBASE_ZERO, ZKE_ASSERT, "begin_tx.py:106-108 access list (coinbase): value_prev == 0") \
  X(EV_BT_AL_CALLER_UNSAT, ZKE_UNSAT, "begin_tx.py:106-108 add_account_to_access_list(caller) unsat") \
  X(EV_BT_AL_CALLER_AMBIG, ZKE_AMBIG, "begin_tx.py:106-108 add_account_to_access_list(caller) ambiguous") \
  X(EV_BT_AL_CALLER_TYPE, ZKE_ASSERT, "begin_tx.py:106-108 access list (caller): value_prev.value() of a Word-typed cell") \
  X(EV_BT_AL_CALLER_ZERO, ZKE_ASSERT, "begin_tx.py:106-108 access list (caller): value_prev == 0") \
  X(EV_BT_AL_CALLEE_UNSAT, ZKE_UNSAT, "begin_tx.py:106-108 add_account_to_access_list(callee) unsat") \
  X(EV_BT_AL_CALLEE_AMBIG, ZKE_AMBIG, "begin_tx.py:106-108 add_account_to_access_list(callee) ambiguous") \
  X(EV_BT_AL_CALLEE_TYPE, ZKE_ASSERT, "begin_tx.py:106-108 access list (callee): value_prev.value() of a Word-typed cell") \
  X(EV_BT_AL_CALLEE_ZERO, ZKE_ASSERT, "begin_tx.py:106-108 access list (callee): value_prev == 0") \
  X(EV_BT_BAL_SENDER_UNSAT, ZKE_UNSAT, "begin_tx.py:111 transfer_with_gas_fee: sub_balance(sender) account_write_word unsat") \
  X(EV_BT_BAL_SENDER_AMBIG, ZKE_AMBIG, "begin_tx.py:111 transfer_with_gas_fee: sub_balance(sender) account_write_word ambiguous") \
  X(EV_BT_BAL_SENDER_REV_UNSAT, ZKE_UNSAT, "begin_tx.py:111 sub_balance(sender): reversion write (instruction.py:848-861) unsat") \
  X(EV_BT_BAL_SENDER_REV_AMBIG, ZKE_AMBIG, "begin_tx.py:111 sub_balance(sender): reversion write (instruction.py:848-861) ambiguous") \
  X(EV_BT_SENDER_EQ, ZKE_ASSERT, "begin_tx.py:111 sub_balance: balance_prev == balance + value + gas_fee (instruction.py:1011)") \
  X(EV_BT_SENDER_CARRY, ZKE_ASSERT, "begin_tx.py:111 sub_balance: carry == 0") \
  X(EV_BT_BAL_RECV_UNSAT, ZKE_UNSAT, "begin_tx.py:111 add_balance(receiver) account_write_word unsat") \
  X(EV_BT_BAL_RECV_AMBIG, ZKE_AMBIG, "begin_tx.py:111 add_balance(receiver) account_write_word ambiguous") \
  X(EV_BT_BAL_RECV_REV_UNSAT, ZKE_UNSAT, "begin_tx.py:111 add_balance(receiver): reversion write unsat") \
  X(EV_BT_BAL_RECV_REV_AMBIG, ZKE_AMBIG, "begin_tx.py:111 add_balance(receiver): reversion write ambiguous") \
  X(EV_BT_RECV_EQ, ZKE_ASSERT, "begin_tx.py:111 add_balance: balance == balance_prev + value") \
  X(EV_BT_RECV_CARRY, ZKE_ASSERT, "begin_tx.py:111 add_balance: carry == 0") \
  X(EV_BT_BALPREV_BYTES, ZKE_VALUE, "begin_tx.py:119-124 word_to_fq(sender_balance_prev, 31): OverflowError") \
  X(EV_BT_BALPREV_RANGE, ZKE_RANGE, "begin_tx.py:119-124 word_to_fq(sender_balance_prev, 31): byte 31 not zero") \
  X(EV_BT_VALUE_BYTES, ZKE_VALUE, "begin_tx.py:119-124 word_to_fq(tx_value, 31): OverflowError") \
  X(EV_BT_VALUE_RANGE, ZKE_RANGE, "begin_tx.py:119-124 word_to_fq(tx_value, 31): byte 31 not zero") \
  X(EV_BT_FEE_BYTES, ZKE_VALUE, "begin_tx.py:119-124 word_to_fq(gas_fee, 31): OverflowError") \
  X(EV_BT_FEE_RANGE, ZKE_RANGE, "begin_tx.py:119-124 word_to_fq(gas_fee, 31): byte 31 not zero") \
  X(EV_BT_BAL_CMP_RANGE, ZKE_ASSERT, "begin_tx.py:119-124 compare(balance_prev, value + gas_fee, 31): operands < 256^31") \
  X(EV_BT_INVALID_FLAG, ZKE_ASSERT, "begin_tx.py:128 is_tx_invalid == invalid_tx") \
  X(EV_BT_PERSISTENT1, ZKE_ASSERT, "begin_tx.py:133 / 234 tx is persistent") \
  X(EV_BT_NEXT_ENDTX, ZKE_ASSERT, "begin_tx.py:136 / 237 next.execution_state == EndTx") \
  X(EV_BT_END_RWC, ZKE_ASSERT, "begin_tx.py:137-140 / 238-241 rw_counter delta") \
  X(EV_BT_END_CALLID, ZKE_ASSERT, "begin_tx.py:137-140 / 238-241 call_id To(call_id)") \
  X(EV_BT_COPY1_UNSAT, ZKE_UNSAT, "begin_tx.py:148-158 copy_lookup(tx calldata -> RlcAcc) unsat") \
  X(EV_BT_COPY1_AMBIG, ZKE_AMBIG, "begin_tx.py:148-158 copy_lookup(tx calldata -> RlcAcc) ambiguous") \
  X(EV_BT_COPY1_RWC0, ZKE_ASSERT, "begin_tx.py:160 assert copy_rwc_inc == 0") \
  X(EV_BT_KECCAK_UNSAT, ZKE_UNSAT, "begin_tx.py:163 keccak_lookup(call_data_length, calldata rlc) unsat") \
  X(EV_BT_KECCAK_AMBIG, ZKE_AMBIG, "begin_tx.py:163 keccak_lookup(call_data_length, calldata rlc) ambiguous") \
  X(EV_BT_COPY2_UNSAT, ZKE_UNSAT, "begin_tx.py:167-177 copy_lookup(tx calldata -> Bytecode) unsat") \
  X(EV_BT_COPY2_AMBIG, ZKE_AMBIG, "begin_tx.py:167-177 copy_lookup(tx calldata -> Bytecode) ambiguous") \
  X(EV_BT_COPY2_RWC0, ZKE_ASSERT, "begin_tx.py:178 assert copy_rwc_inc == 0") \
  X(EV_BT_PRECOMPILE, ZKE_NOTIMPL, "begin_tx.py:225-227 callee is a precompile: raise NotImplementedError") \
  X(EV_BT_ACC_CODEHASH_UNSAT, ZKE_UNSAT, "begin_tx.py:229 account_read_word(callee, CodeHash) unsat") \
  X(EV_BT_ACC_CODEHASH_AMBIG, ZKE_AMBIG, "begin_tx.py:229 account_read_word(callee, CodeHash) ambiguous") \
  X(EV_BT_CTX0_UNSAT, ZKE_UNSAT, "begin_tx.py:183-201 / 250-269 call_context_lookup_word(Depth) unsat") \
  X(EV_BT_CTX0_AMBIG, ZKE_AMBIG, "begin_tx.py:183-201 / 250-269 call_context_lookup_word(Depth) ambiguous") \
  X(EV_BT_CTX0_EQ, ZKE_ASSERT, "begin_tx.py:198-201 / 266-269 call context Depth == expected") \
  X(EV_BT_CTX1_UNSAT, ZKE_UNSAT, "begin_tx.py:183-201 / 250-269 call_context_lookup_word(CallerAddress) unsat") \
  X(EV_BT_CTX1_AMBIG, ZKE_AMBIG, "begin_tx.py:183-201 / 250-269 call_context_lookup_word(CallerAddress) ambiguous") \
  X(EV_BT_CTX1_EQ, ZKE_ASSERT, "begin_tx.py:198-201 / 266-269 call context CallerAddress == expected") \
  X(EV_BT_CTX2_UNSAT, ZKE_UNSAT, "begin_tx.py:183-201 / 250-269 call_context_lookup_word(CalleeAddress) unsat") \
  X(EV_BT_CTX2_AMBIG, ZKE_AMBIG, "begin_tx.py:183-201 / 250-269 call_context_lookup_word(CalleeAddress) ambiguous") \
  X(EV_BT_CTX2_EQ, ZKE_ASSERT, "begin_tx.py:198-201 / 266-269 call context CalleeAddress == expected") \
  X(EV_BT_CTX3_UNSAT, ZKE_UNSAT, "begin_tx.py:183-201 / 250-269 call_context_lookup_word(CallDataOffset) unsat") \
  X(EV_BT_CTX3_AMBIG, ZKE_AMBIG, "begin_tx.py:183-201 / 250-269 call_context_lookup_word(CallDataOffset) ambiguous") \
  X(EV_BT_CTX3_EQ, ZKE_ASSERT, "begin_tx.py:198-201 / 266-269 call context CallDataOffset == expected") \
  X(EV_BT_CTX4_UNSAT, ZKE_UNSAT, "begin_tx.py:183-201 / 250-269 call_context_lookup_word(CallDataLength) unsat") \
  X(EV_BT_CTX4_AMBIG, ZKE_AMBIG, "begin_tx.py:183-201 / 250-269 call_context_lookup_word(CallDataLength) ambiguous") \
  X(EV_BT_CTX4_EQ, ZKE_ASSERT, "begin_tx.py:198-201 / 266-269 call context CallDataLength == expected") \
  X(EV_BT_CTX5_UNSAT, ZKE_UNSAT, "begin_tx.py:183-201 / 250-269 call_context_lookup_word(Value) unsat") \
  X(EV_BT_CTX5_AMBIG, ZKE_AMBIG, "begin_tx.py:183-201 / 250-269 call_context_lookup_word(Value) ambiguous") \
  X(EV_BT_CTX5_EQ, ZKE_ASSERT, "begin_tx.py:198-201 / 266-269 call context Value == expected") \
  X(EV_BT_CTX6_UNSAT, ZKE_UNSAT, "begin_tx.py:183-201 / 250-269 call_context_lookup_word(IsStatic) unsat") \
  X(EV_BT_CTX6_AMBIG, ZKE_AMBIG, "begin_tx.py:183-201 / 250-269 call_context_lookup_word(IsStatic) ambiguous") \
  X(EV_BT_CTX6_EQ, ZKE_ASSERT, "begin_tx.py:198-201 / 266-269 call context IsStatic == expected") \
  X(EV_BT_CTX7_UNSAT, ZKE_UNSAT, "begin_tx.py:183-201 / 250-269 call_context_lookup_word(LastCalleeId) unsat") \
  X(EV_BT_CTX7_AMBIG, ZKE_AMBIG, "begin_tx.py:183-201 / 250-269 call_context_lookup_word(LastCalleeId) ambiguous") \
  X(EV_BT_CTX7_EQ, ZKE_ASSERT, "begin_tx.py:198-201 / 266-269 call context LastCalleeId == expected") \
  X(EV_BT_CTX8_UNSAT, ZKE_UNSAT, "begin_tx.py:183-201 / 250-269 call_context_lookup_word(LastCalleeReturnDataOffset) unsat") \
  X(EV_BT_CTX8_AMBIG, ZKE_AMBIG, "begin_tx.py:183-201 / 250-269 call_context_lookup_word(LastCalleeReturnDataOffset) ambiguous") \
  X(EV_BT_CTX8_EQ, ZKE_ASSERT, "begin_tx.py:198-201 / 266-269 call context LastCalleeReturnDataOffset == expected") \
  X(EV_BT_CTX9_UNSAT, ZKE_UNSAT, "begin_tx.py:183-201 / 250-269 call_context_lookup_word(LastCalleeReturnDataLength) unsat") \
  X(EV_BT_CTX9_AMBIG, ZKE_AMBIG, "begin_tx.py:183-201 / 250-269 call_context_lookup_word(LastCalleeReturnDataLength) ambiguous") \
  X(EV_BT_CTX9_EQ, ZKE_ASSERT, "begin_tx.py:198-201 / 266-269 call context LastCalleeReturnDataLength == expected") \
  X(EV_BT_CTX10_UNSAT, ZKE_UNSAT, "begin_tx.py:183-201 / 250-269 call_context_lookup_word(IsRoot) unsat") \
  X(EV_BT_CTX10_AMBIG, ZKE_AMBIG, "begin_tx.py:183-201 / 250-269 call_context_lookup_word(IsRoot) ambiguous") \
  X(EV_BT_CTX10_EQ, ZKE_ASSERT, "begin_tx.py:198-201 / 266-269 call context IsRoot == expected") \
  X(EV_BT_CTX11_UNSAT, ZKE_UNSAT, "begin_tx.py:183-201 / 250-269 call_context_lookup_word(IsCreate) unsat") \
  X(EV_BT_CTX11_AMBIG, ZKE_AMBIG, "begin_tx.py:183-201 / 250-269 call_context_lookup_word(IsCreate) ambiguous") \
  X(EV_BT_CTX11_EQ, ZKE_ASSERT, "begin_tx.py:198-201 / 266-269 call context IsCreate == expected") \
  X(EV_BT_CTX12_UNSAT, ZKE_UNSAT, "begin_tx.py:183-201 / 250-269 call_context_lookup_word(CodeHash) unsat") \
  X(EV_BT_CTX12_AMBIG, ZKE_AMBIG, "begin_tx.py:183-201 / 250-269 call_context_lookup_word(CodeHash) ambiguous") \
  X(EV_BT_CTX12_EQ, ZKE_ASSERT, "begin_tx.py:198-201 / 266-269 call context CodeHash == expected") \
  X(EV_BT_NC_RWC, ZKE_ASSERT, "begin_tx.py:203-212 / 271-280 step_state_transition_to_new_context: RWC (instruction.py:266-290)") \
  X(EV_BT_NC_CALL_ID, ZKE_ASSERT, "begin_tx.py:203-212 / 271-280 step_state_transition_to_new_context: CALL_ID (instruction.py:266-290)") \
  X(EV_BT_NC_IS_ROOT, ZKE_ASSERT, "begin_tx.py:203-212 / 271-280 step_state_transition_to_new_context: IS_ROOT (instruction.py:266-290)") \
  X(EV_BT_NC_IS_CREATE, ZKE_ASSERT, "begin_tx.py:203-212 / 271-280 step_state_transition_to_new_context: IS_CREATE (instruction.py:266-290)") \
  X(EV_BT_NC_CODE_HASH, ZKE_ASSERT, "begin_tx.py:203-212 / 271-280 step_state_transition_to_new_context: CODE_HASH (instruction.py:266-290)") \
  X(EV_BT_NC_GAS_LEFT, ZKE_ASSERT, "begin_tx.py:203-212 / 271-280 step_state_transition_to_new_context: GAS_LEFT (instruction.py:266-290)") \
  X(EV_BT_NC_REV, ZKE_ASSERT, "begin_tx.py:203-212 / 271-280 step_state_transition_to_new_context: REV (instruction.py:266-290)") \
  X(EV_BT_NC_LOG_ID, ZKE_ASSERT, "begin_tx.py:203-212 / 271-280 step_state_transition_to_new_context: LOG_ID (instruction.py:266-290)") \
  X(EV_BT_NC_PC, ZKE_ASSERT, "begin_tx.py:203-212 / 271-280 step_state_transition_to_new_context: PC (instruction.py:266-290)") \
  X(EV_BT_NC_SP, ZKE_ASSERT, "begin_tx.py:203-212 / 271-280 step_state_transition_to_new_context: SP (instruction.py:266-290)") \
  X(EV_BT_NC_MEM, ZKE_ASSERT, "begin_tx.py:203-212 / 271-280 step_state_transition_to_new_context: MEM (instruction.py:266-290)") \
  /* error states: the shared tail constrain_error_state (instruction.py:1426-1452); the restore-to-caller branch \
   * reports through the EV_RST* ids */                                                                         \
  X(EV_ERR_CC_UNSAT, ZKE_UNSAT, "instruction.py:1429 call_context_lookup(IsSuccess) unsat")                      \
  X(EV_ERR_CC_AMBIG, ZKE_AMBIG, "instruction.py:1429 call_context_lookup(IsSuccess) ambiguous")                  \
  X(EV_ERR_CC_TYPE, ZKE_ASSERT, "instruction.py:1429 .value(): IsSuccess is a Word")                             \
  X(EV_ERR_IS_SUCCESS, ZKE_ASSERT, "instruction.py:1430 is_success == 0")                                        \
  X(EV_ERR_ROOT_ENDTX, ZKE_ASSERT, "instruction.py:1433-1434 is_root == (next state is EndTx)")                  \
  X(EV_ERR_RWC, ZKE_ASSERT, "instruction.py:1439-1442 root: rw_counter + rw lookups + reversible_write_counter + 1") \
  X(EV_ERR_CALL_ID, ZKE_ASSERT, "instruction.py:1439-1442 root: call_id same")                                   \
  X(EV_ESTK_RESP_OPCODE, ZKE_UNSAT, "error_stack.py:7 responsible_opcode_lookup(opcode, stack_pointer)")         \
  X(EV_EINV_RESP_OPCODE, ZKE_UNSAT, "error_invalid_opcode.py:8 responsible_opcode_lookup(opcode)")               \
  X(EV_EOGC_OPCODE_VALUE, ZKE_VALUE, "error_oog_constant.py:11 Opcode(opcode.n): not a valid opcode -> ValueError") \
  X(EV_EOGC_GAS_UNSAT, ZKE_UNSAT, "error_oog_constant.py:10-12 fixed_lookup(OpcodeConstantGas, opcode, gas)")    \
  X(EV_EOGC_CMP_RANGE, ZKE_ASSERT, "error_oog_constant.py:15-17 compare(): operand exceeds 8 bytes")             \
  X(EV_EOGC_NOT_ENOUGH, ZKE_ASSERT, "error_oog_constant.py:18 gas_left < constant gas")                          \
  X(EV_EJMP_OPCODE, ZKE_ASSERT, "error_invalid_jump.py:10 opcode in (JUMP, JUMPI)")                              \
  X(EV_EJMP_LEN_UNSAT, ZKE_UNSAT, "error_invalid_jump.py:12 bytecode_length lookup unsat")                       \
  X(EV_EJMP_LEN_AMBIG, ZKE_AMBIG, "error_invalid_jump.py:12 bytecode_length lookup ambiguous")                   \
  X(EV_EJMP_DEST_UNSAT, ZKE_UNSAT, "error_invalid_jump.py:13 stack_pop(dest) unsat")                             \
  X(EV_EJMP_DEST_AMBIG, ZKE_AMBIG, "error_invalid_jump.py:13 stack_pop(dest) ambiguous")                         \
  X(EV_EJMP_COND_UNSAT, ZKE_UNSAT, "error_invalid_jump.py:16 stack_pop(condition) unsat")                        \
  X(EV_EJMP_COND_AMBIG, ZKE_AMBIG, "error_invalid_jump.py:16 stack_pop(condition) ambiguous")                    \
  X(EV_EJMP_COND_ZERO, ZKE_ASSERT, "error_invalid_jump.py:18 condition != 0")                                    \
  X(EV_EJMP_DEST_DOMAIN, ZKE_VALUE, "error_invalid_jump.py:20 word_to_u64: to_le_bytes of a half >= 2^128 -> OverflowError") \
  X(EV_EJMP_DEST_U64, ZKE_RANGE, "error_invalid_jump.py:20 word_to_u64(dest): more than 8 bytes")                \
  X(EV_EJMP_CMP_RANGE, ZKE_ASSERT, "error_invalid_jump.py:22 compare(): code length exceeds 8 bytes")            \
  X(EV_EJMP_AT_UNSAT, ZKE_UNSAT, "error_invalid_jump.py:26 bytecode_lookup_pair(dest) unsat")                    \
  X(EV_EJMP_AT_AMBIG, ZKE_AMBIG, "error_invalid_jump.py:26 bytecode_lookup_pair(dest) ambiguous")                \
  X(EV_EJMP_IS_JUMPDEST, ZKE_ASSERT, "error_invalid_jump.py:28-29 is_code * (value == JUMPDEST) == 0")           \
  /* selfbalance.py */                                                                                          \
  X(EV_SBAL_OPCODE, ZKE_ASSERT, "selfbalance.py:8 opcode == SELFBALANCE")                                        \
  X(EV_SBAL_CC_UNSAT, ZKE_UNSAT, "selfbalance.py:10 call_context_lookup_word(CalleeAddress) unsat")              \
  X(EV_SBAL_CC_AMBIG, ZKE_AMBIG, "selfbalance.py:10 call_context_lookup_word(CalleeAddress) ambiguous")          \
  X(EV_SBAL_ADDR_DOMAIN, ZKE_VALUE, "selfbalance.py:11 word_to_address: to_le_bytes of a half >= 2^128 -> OverflowError") \
  X(EV_SBAL_ADDR_RANGE, ZKE_RANGE, "selfbalance.py:11 word_to_address: more than 20 bytes")                      \
  X(EV_SBAL_ACC_UNSAT, ZKE_UNSAT, "selfbalance.py:12 account_read_word(Balance) unsat")                          \
  X(EV_SBAL_ACC_AMBIG, ZKE_AMBIG, "selfbalance.py:12 account_read_word(Balance) ambiguous")                      \
  X(EV_SBAL_PUSH_UNSAT, ZKE_UNSAT, "selfbalance.py:13 stack_push unsat")                                         \
  X(EV_SBAL_PUSH_AMBIG, ZKE_AMBIG, "selfbalance.py:13 stack_push ambiguous")                                     \
  X(EV_SBAL_EQ, ZKE_ASSERT, "selfbalance.py:13 pushed word == balance")                                          \
  /* out-of-gas / out-of-bound error states (error_oog_sha3.py, error_oog_static_memory_expansion.py,            \
   * error_oog_dynamic_memory_expansion.py, error_oog_log.py, error_oog_exp.py, error_return_data_out_of_bound.py): \
   * one id per KIND of constraint, shared by the six gate programs (a step reports one id; its state names the file) */ \
  X(EV_EOOG_OPCODE, ZKE_ASSERT, "error_oog_*.py / error_return_data_out_of_bound.py: the opcode is not one the state is responsible for") \
  X(EV_EOOG_LOG_RANGE5, ZKE_UNSAT, "error_oog_log.py:12 range_lookup(opcode - LOG0, 5)")                          \
  X(EV_EOOG_POP0_UNSAT, ZKE_UNSAT, "first stack lookup of the error state unsat")                                \
  X(EV_EOOG_POP0_AMBIG, ZKE_AMBIG, "first stack lookup of the error state ambiguous")                            \
  X(EV_EOOG_POP1_UNSAT, ZKE_UNSAT, "second stack lookup of the error state unsat")                               \
  X(EV_EOOG_POP1_AMBIG, ZKE_AMBIG, "second stack lookup of the error state ambiguous")                           \
  X(EV_EOOG_W0_DOMAIN, ZKE_VALUE, "word_to_fq / byte_size of the first word: to_le_bytes of a half >= 2^128 -> OverflowError") \
  X(EV_EOOG_W0_RANGE, ZKE_RANGE, "word_to_fq of the first word: too many bytes (instruction.py:480-484)")        \
  X(EV_EOOG_W1_DOMAIN, ZKE_VALUE, "word_to_fq of the second word: to_le_bytes of a half >= 2^128 -> OverflowError") \
  X(EV_EOOG_W1_RANGE, ZKE_RANGE, "word_to_fq of the second word: too many bytes")                                \
  X(EV_EOOG_MEMSIZE_RANGE, ZKE_RANGE, "memory_expansion[_dynamic_length]: memory size exceeds 4 bytes (instruction.py:1139-1145, 1164-1166)") \
  X(EV_EOOG_MEM_MAX, ZKE_ASSERT, "memory_expansion[_dynamic_length]: max(): curr.memory_word_size exceeds 4 bytes") \
  X(EV_EOOG_WORDSIZE_RANGE, ZKE_RANGE, "error_oog_sha3.py:24-26 minimum_word_size exceeds 4 bytes")              \
  X(EV_EOOG_CC_UNSAT, ZKE_UNSAT, "error_return_data_out_of_bound.py:16-18 call_context_lookup(LastCalleeReturnDataLength) unsat") \
  X(EV_EOOG_CC_AMBIG, ZKE_AMBIG, "error_return_data_out_of_bound.py:16-18 call_context_lookup ambiguous")        \
  X(EV_EOOG_CC_TYPE, ZKE_ASSERT, "error_return_data_out_of_bound.py:16-18 .value(): the cell is a Word")         \
  X(EV_EOOG_CMP_RANGE, ZKE_ASSERT, "compare(): an operand exceeds n_bytes (8: gas; 31: return data end)")        \
  X(EV_EOOG_NOT_ENOUGH, ZKE_ASSERT, "gas_left < required gas / no out-of-bound condition holds")                  \
  /* BALANCE / EXTCODEHASH / EXTCODESIZE (balance.py, extcodehash.py, extcodesize.py) and                         \
   * ErrorOutOfGasAccountAccess (error_oog_account_access.py): shared ids, one per kind of constraint */         \
  X(EV_ACC_OPCODE, ZKE_ASSERT, "balance.py:9 / extcodehash.py:9 / extcodesize.py:14 / error_oog_account_access.py:25 opcode") \
  X(EV_ACC_POP_UNSAT, ZKE_UNSAT, "stack_pop(address) unsat")                                                     \
  X(EV_ACC_POP_AMBIG, ZKE_AMBIG, "stack_pop(address) ambiguous")                                                 \
  X(EV_ACC_ADDR_DOMAIN, ZKE_VALUE, "word_to_address: to_le_bytes of a half >= 2^128 -> OverflowError")           \
  X(EV_ACC_ADDR_RANGE, ZKE_RANGE, "word_to_address: more than 20 bytes")                                         \
  X(EV_ACC_TXID_UNSAT, ZKE_UNSAT, "call_context_lookup(TxId) unsat")                                             \
  X(EV_ACC_TXID_AMBIG, ZKE_AMBIG, "call_context_lookup(TxId) ambiguous")                                         \
  X(EV_ACC_TXID_TYPE, ZKE_ASSERT, "call_context_lookup(TxId).value(): the cell is a Word")                       \
  X(EV_ACC_REVEND_UNSAT, ZKE_UNSAT, "reversion_info: call_context_lookup(RwCounterEndOfReversion) unsat")        \
  X(EV_ACC_REVEND_AMBIG, ZKE_AMBIG, "reversion_info: RwCounterEndOfReversion ambiguous")                         \
  X(EV_ACC_REVEND_TYPE, ZKE_ASSERT, "reversion_info: RwCounterEndOfReversion is a Word")                         \
  X(EV_ACC_PERSIST_UNSAT, ZKE_UNSAT, "reversion_info: call_context_lookup(IsPersistent) unsat")                  \
  X(EV_ACC_PERSIST_AMBIG, ZKE_AMBIG, "reversion_info: IsPersistent ambiguous")                                   \
  X(EV_ACC_PERSIST_TYPE, ZKE_ASSERT, "reversion_info: IsPersistent is a Word")                                   \
  X(EV_ACC_AL_UNSAT, ZKE_UNSAT, "add_account_to_access_list / read_account_to_access_list: rw lookup unsat (instruction.py:1044-1069)") \
  X(EV_ACC_AL_AMBIG, ZKE_AMBIG, "add_account_to_access_list / read_account_to_access_list: rw lookup ambiguous")  \
  X(EV_ACC_AL_REV_UNSAT, ZKE_UNSAT, "state_write: the reversion row is missing (instruction.py:848-861)")        \
  X(EV_ACC_AL_REV_AMBIG, ZKE_AMBIG, "state_write: the reversion row is ambiguous")                               \
  X(EV_ACC_AL_PREV_TYPE, ZKE_ASSERT, "access list row: value_prev.value(): the cell is a Word")                  \
  X(EV_ACC_HASH_UNSAT, ZKE_UNSAT, "account_read_word(CodeHash) unsat")                                           \
  X(EV_ACC_HASH_AMBIG, ZKE_AMBIG, "account_read_word(CodeHash) ambiguous")                                       \
  X(EV_ACC_BAL_UNSAT, ZKE_UNSAT, "balance.py:23 account_read_word(Balance) unsat")                               \
  X(EV_ACC_BAL_AMBIG, ZKE_AMBIG, "balance.py:23 account_read_word(Balance) ambiguous")                           \
  X(EV_ACC_LEN_UNSAT, ZKE_UNSAT, "extcodesize.py:26 bytecode_length(code_hash) unsat")                           \
  X(EV_ACC_LEN_AMBIG, ZKE_AMBIG, "extcodesize.py:26 bytecode_length(code_hash) ambiguous")                       \
  X(EV_ACC_SIZE_WORD, ZKE_ASSERT, "extcodesize.py:31 Word.from_lo(code_size): code_size >= 2^128")               \
  X(EV_ACC_PUSH_UNSAT, ZKE_UNSAT, "stack_push unsat")                                                            \
  X(EV_ACC_PUSH_AMBIG, ZKE_AMBIG, "stack_push ambiguous")                                                        \
  X(EV_ACC_EQ, ZKE_ASSERT, "the pushed word == balance / code hash / code size")                                 \
  X(EV_ACC_WARM_BOOL, ZKE_ASSERT, "instruction.py:422 select(is_warm, ..): the access-list value_prev is not 0 / 1") \
  /* CODECOPY / RETURNDATACOPY / EXTCODECOPY (codecopy.py, returndatacopy.py, extcodecopy.py) and                  \
   * ErrorOutOfGasMemoryCopy (error_oog_memory_copy.py): shared ids, one per kind of constraint */               \
  X(EV_CPY_OPCODE, ZKE_ASSERT, "error_oog_memory_copy.py:28-30 opcode is one of the four copy opcodes")          \
  X(EV_CPY_POP0_UNSAT, ZKE_UNSAT, "stack lookup 0 unsat")                                                        \
  X(EV_CPY_POP0_AMBIG, ZKE_AMBIG, "stack lookup 0 ambiguous")                                                    \
  X(EV_CPY_POP1_UNSAT, ZKE_UNSAT, "stack lookup 1 unsat")                                                        \
  X(EV_CPY_POP1_AMBIG, ZKE_AMBIG, "stack lookup 1 ambiguous")                                                    \
  X(EV_CPY_POP2_UNSAT, ZKE_UNSAT, "stack lookup 2 unsat")                                                        \
  X(EV_CPY_POP2_AMBIG, ZKE_AMBIG, "stack lookup 2 ambiguous")                                                    \
  X(EV_CPY_POP3_UNSAT, ZKE_UNSAT, "stack lookup 3 unsat")                                                        \
  X(EV_CPY_POP3_AMBIG, ZKE_AMBIG, "stack lookup 3 ambiguous")                                                    \
  X(EV_CPY_ADDR_DOMAIN, ZKE_VALUE, "word_to_address / word_to_fq(external address): OverflowError")              \
  X(EV_CPY_ADDR_RANGE, ZKE_RANGE, "word_to_address (20 bytes; 5 bytes in error_oog_memory_copy.py:45): too many bytes") \
  X(EV_CPY_SIZE_DOMAIN, ZKE_VALUE, "memory_offset_and_length: word_to_fq(size): OverflowError")                  \
  X(EV_CPY_SIZE_RANGE, ZKE_RANGE, "memory_offset_and_length: size exceeds 5 bytes")                              \
  X(EV_CPY_MOFF_DOMAIN, ZKE_VALUE, "memory_offset_and_length: word_to_fq(memory offset): OverflowError")         \
  X(EV_CPY_MOFF_RANGE, ZKE_RANGE, "memory_offset_and_length: memory offset exceeds 5 bytes")                     \
  X(EV_CPY_OFF_DOMAIN, ZKE_VALUE, "word_to_fq(code / data offset): OverflowError")                               \
  X(EV_CPY_OFF_RANGE, ZKE_RANGE, "code offset exceeds 5 bytes (codecopy.py:16) / 8 bytes (extcodecopy.py:15, returndatacopy.py:26)") \
  X(EV_CPY_SIZE8_DOMAIN, ZKE_VALUE, "returndatacopy.py:26 word_to_fq(size, 8): OverflowError")                   \
  X(EV_CPY_SIZE8_RANGE, ZKE_RANGE, "returndatacopy.py:26 size exceeds 8 bytes")                                  \
  X(EV_CPY_LEN_UNSAT, ZKE_UNSAT, "codecopy.py:18 bytecode_length(curr.code_hash) unsat")                         \
  X(EV_CPY_LEN_AMBIG, ZKE_AMBIG, "codecopy.py:18 bytecode_length ambiguous")                                     \
  X(EV_CPY_CC0_UNSAT, ZKE_UNSAT, "returndatacopy.py:15 call_context_lookup(LastCalleeId) unsat")                 \
  X(EV_CPY_CC0_AMBIG, ZKE_AMBIG, "returndatacopy.py:15 LastCalleeId ambiguous")                                  \
  X(EV_CPY_CC0_TYPE, ZKE_ASSERT, "returndatacopy.py:15 LastCalleeId is a Word")                                  \
  X(EV_CPY_CC1_UNSAT, ZKE_UNSAT, "returndatacopy.py:16-18 call_context_lookup(LastCalleeReturnDataLength) unsat") \
  X(EV_CPY_CC1_AMBIG, ZKE_AMBIG, "returndatacopy.py:16-18 LastCalleeReturnDataLength ambiguous")                 \
  X(EV_CPY_CC1_TYPE, ZKE_ASSERT, "returndatacopy.py:16-18 LastCalleeReturnDataLength is a Word")                 \
  X(EV_CPY_CC2_UNSAT, ZKE_UNSAT, "returndatacopy.py:19-21 call_context_lookup(LastCalleeReturnDataOffset) unsat") \
  X(EV_CPY_CC2_AMBIG, ZKE_AMBIG, "returndatacopy.py:19-21 LastCalleeReturnDataOffset ambiguous")                 \
  X(EV_CPY_CC2_TYPE, ZKE_ASSERT, "returndatacopy.py:19-21 LastCalleeReturnDataOffset is a Word")                 \
  X(EV_CPY_OOB_RANGE, ZKE_RANGE, "returndatacopy.py:24-28 range_check(return_data_length - (offset + size), 4)") \
  X(EV_CPY_MEMSIZE_RANGE, ZKE_RANGE, "memory_expansion_dynamic_length: memory size exceeds 4 bytes")             \
  X(EV_CPY_MEM_MAX, ZKE_ASSERT, "memory_expansion_dynamic_length: max(): curr.memory_word_size exceeds 4 bytes") \
  X(EV_CPY_WORDSIZE_RANGE, ZKE_RANGE, "memory_copier_gas_cost: word size exceeds 4 bytes")                       \
  X(EV_CPY_GASCOST_RANGE, ZKE_RANGE, "memory_copier_gas_cost: gas cost exceeds 8 bytes")                         \
  X(EV_CPY_COPY_UNSAT, ZKE_UNSAT, "copy_lookup unsat")                                                           \
  X(EV_CPY_COPY_AMBIG, ZKE_AMBIG, "copy_lookup ambiguous")                                                       \
  X(EV_CPY_RWC_INC, ZKE_ASSERT, "returndatacopy.py:48 copy_rwc_inc == size * 2")                 \
  X(EV_AR_OPCODE, ZKE_ASSERT, "addmod.py:23 / mulmod.py:33 opcode == ADDMOD / MULMOD")            \
  X(EV_AR_RW0_UNSAT, ZKE_UNSAT, "addmod / mulmod / sdiv_smod / sar: 1st stack lookup unsat")       \
  X(EV_AR_RW0_AMBIG, ZKE_AMBIG, "1st stack lookup ambiguous")                                      \
  X(EV_AR_RW1_UNSAT, ZKE_UNSAT, "2nd stack lookup unsat")                                          \
  X(EV_AR_RW1_AMBIG, ZKE_AMBIG, "2nd stack lookup ambiguous")                                      \
  X(EV_AR_RW2_UNSAT, ZKE_UNSAT, "3rd stack lookup unsat")                                          \
  X(EV_AR_RW2_AMBIG, ZKE_AMBIG, "3rd stack lookup ambiguous")                                      \
  X(EV_AR_RW3_UNSAT, ZKE_UNSAT, "4th stack lookup unsat")                                          \
  X(EV_AR_RW3_AMBIG, ZKE_AMBIG, "4th stack lookup ambiguous")                                      \
  X(EV_AR_WITNESS_DOMAIN, ZKE_NOTIMPL, "ADDMOD / MULMOD / SDIV / SMOD witness derivation with a stack word half >= 2^128: outside the supported witness domain (DESIGN.md)") \
  X(EV_AR_ADDMOD_ZERO, ZKE_ASSERT, "addmod.py:60 n == 0 => pushed result == 0")                   \
  X(EV_AR_ADDMOD_CARRY0, ZKE_RANGE, "addmod.py:47-50 mul_add_words_512: range_check(carry_0, 9), instruction.py:658") \
  X(EV_AR_ADDMOD_CARRY1, ZKE_RANGE, "addmod.py:47-50 mul_add_words_512: range_check(carry_1, 9), instruction.py:659") \
  X(EV_AR_MULMOD_R, ZKE_ASSERT, "mulmod.py:56 a_reduced * b == k * n + r")                         \
  X(EV_AR_MULMOD_TO64, ZKE_VALUE, "mulmod.py:62 mul_add_words_512: to_64s(b) with a half >= 2^128 -> OverflowError (n == 0)") \
  X(EV_AR_SDIV_REM_NEG, ZKE_VALUE, "sdiv_smod.py:100 Word(negative int) -> OverflowError")         \
  X(EV_AR_SDIV_REM_WORD, ZKE_ASSERT, "sdiv_smod.py:102 Word(get_int_neg(negative int)) >= 2^256")  \
  X(EV_AR_SDIV_CARRY_LO, ZKE_RANGE, "sdiv_smod.py:50 mul_add_words: range_check(carry_lo, 9)")     \
  X(EV_AR_SDIV_CARRY_HI, ZKE_RANGE, "sdiv_smod.py:50 mul_add_words: range_check(carry_hi, 9)")     \
  X(EV_AR_SDIV_OVERFLOW, ZKE_ASSERT, "sdiv_smod.py:52 overflow == 0")                              \
  X(EV_AR_SDIV_REM_LT, ZKE_ASSERT, "sdiv_smod.py:55-56 |remainder| < |divisor| unless divisor == 0") \
  X(EV_AR_SDIV_SIGN_REM, ZKE_ASSERT, "sdiv_smod.py:60-61 sign(dividend) == sign(remainder)")       \
  X(EV_AR_SDIV_SIGN_QUOT, ZKE_ASSERT, "sdiv_smod.py:72-76 sign(dividend) == sign(divisor) ^ sign(quotient)") \
  X(EV_AR_SAR_BYTES, ZKE_VALUE, "sar.py:57-59,156 to_le_bytes / to_64s: a half >= 2^128 -> OverflowError") \
  X(EV_AR_SAR_RESULT, ZKE_ASSERT, "sar.py:79-82 b64s[idx] == limb of the pushed word")             \
  X(EV_AR_SAR_SIGN_UNSAT, ZKE_UNSAT, "sar.py:142 sign_byte_lookup unsat")                          \
  X(EV_AR_SAR_SIGN_AMBIG, ZKE_AMBIG, "sar.py:142 sign_byte_lookup ambiguous")                      \
  X(EV_AR_SAR_POW_LO_UNSAT, ZKE_UNSAT, "sar.py:151 pow2_lookup(shf_mod64, p_lo) unsat")            \
  X(EV_AR_SAR_POW_LO_AMBIG, ZKE_AMBIG, "sar.py:151 pow2_lookup ambiguous")                         \
  X(EV_AR_SAR_POW_HI_UNSAT, ZKE_UNSAT, "sar.py:152 pow2_lookup(64 - shf_mod64, p_hi) unsat")       \
  X(EV_AR_SAR_POW_HI_AMBIG, ZKE_AMBIG, "sar.py:152 pow2_lookup ambiguous")                 \
  X(EV_ST_OPCODE, ZKE_ASSERT, "storage.py:18,53 opcode == SLOAD / SSTORE")                           \
  X(EV_ST_TXID_UNSAT, ZKE_UNSAT, "storage.py:20,55 call_context_lookup(TxId) unsat")                 \
  X(EV_ST_TXID_AMBIG, ZKE_AMBIG, "storage.py:20,55 call_context_lookup(TxId) ambiguous")             \
  X(EV_ST_TXID_TYPE, ZKE_ASSERT, "storage.py:20,55 call_context_lookup(TxId): .value() of a Word")   \
  X(EV_ST_STATIC_UNSAT, ZKE_UNSAT, "storage.py:57-59 call_context_lookup(IsStatic) unsat")           \
  X(EV_ST_STATIC_AMBIG, ZKE_AMBIG, "storage.py:57-59 call_context_lookup(IsStatic) ambiguous")       \
  X(EV_ST_STATIC_TYPE, ZKE_ASSERT, "storage.py:57-59 call_context_lookup(IsStatic): .value() of a Word") \
  X(EV_ST_STATIC_NONZERO, ZKE_ASSERT, "storage.py:57-59 IsStatic == 0")                              \
  X(EV_ST_REVEND_UNSAT, ZKE_UNSAT, "reversion_info: call_context_lookup(RwCounterEndOfReversion) unsat") \
  X(EV_ST_REVEND_AMBIG, ZKE_AMBIG, "reversion_info: call_context_lookup(RwCounterEndOfReversion) ambiguous") \
  X(EV_ST_REVEND_TYPE, ZKE_ASSERT, "reversion_info: call_context_lookup(RwCounterEndOfReversion): .value() of a Word") \
  X(EV_ST_PERSIST_UNSAT, ZKE_UNSAT, "reversion_info: call_context_lookup(IsPersistent) unsat")       \
  X(EV_ST_PERSIST_AMBIG, ZKE_AMBIG, "reversion_info: call_context_lookup(IsPersistent) ambiguous")   \
  X(EV_ST_PERSIST_TYPE, ZKE_ASSERT, "reversion_info: call_context_lookup(IsPersistent): .value() of a Word") \
  X(EV_ST_CALLEE_UNSAT, ZKE_UNSAT, "storage.py:22,62 call_context_lookup_word(CalleeAddress) unsat") \
  X(EV_ST_CALLEE_AMBIG, ZKE_AMBIG, "storage.py:22,62 call_context_lookup_word(CalleeAddress) ambiguous") \
  X(EV_ST_CALLEE_DOMAIN, ZKE_VALUE, "word_to_address: to_le_bytes of a half >= 2^128 -> OverflowError") \
  X(EV_ST_CALLEE_RANGE, ZKE_RANGE, "word_to_address: more than 20 bytes")                            \
  X(EV_ST_KEY_UNSAT, ZKE_UNSAT, "storage.py:25,65 stack_pop storage key unsat")                      \
  X(EV_ST_KEY_AMBIG, ZKE_AMBIG, "storage.py:25,65 stack_pop storage key ambiguous")                  \
  X(EV_ST_VAL_UNSAT, ZKE_UNSAT, "storage.py:66 stack_pop storage value unsat")                       \
  X(EV_ST_VAL_AMBIG, ZKE_AMBIG, "storage.py:66 stack_pop storage value ambiguous")                   \
  X(EV_ST_READ_UNSAT, ZKE_UNSAT, "storage.py:28 account_storage_read unsat")                         \
  X(EV_ST_READ_AMBIG, ZKE_AMBIG, "storage.py:28 account_storage_read ambiguous")                     \
  X(EV_ST_PUSH_UNSAT, ZKE_UNSAT, "storage.py:29 stack_push unsat")                                   \
  X(EV_ST_PUSH_AMBIG, ZKE_AMBIG, "storage.py:29 stack_push ambiguous")                               \
  X(EV_ST_READ_EQ, ZKE_ASSERT, "storage.py:27-30 storage value == pushed word")                      \
  X(EV_ST_WRITE_UNSAT, ZKE_UNSAT, "storage.py:67-72 account_storage_write unsat")                    \
  X(EV_ST_WRITE_AMBIG, ZKE_AMBIG, "storage.py:67-72 account_storage_write ambiguous")                \
  X(EV_ST_WRITE_REV_UNSAT, ZKE_UNSAT, "storage.py:67-72 account_storage_write: reversion row unsat") \
  X(EV_ST_WRITE_REV_AMBIG, ZKE_AMBIG, "storage.py:67-72 account_storage_write: reversion row ambiguous") \
  X(EV_ST_WRITE_EQ, ZKE_ASSERT, "storage.py:73 popped value == written value")                       \
  X(EV_ST_AL_UNSAT, ZKE_UNSAT, "storage.py:32-37,75-80 add_account_storage_to_access_list unsat")    \
  X(EV_ST_AL_AMBIG, ZKE_AMBIG, "storage.py:32-37,75-80 add_account_storage_to_access_list ambiguous") \
  X(EV_ST_AL_REV_UNSAT, ZKE_UNSAT, "add_account_storage_to_access_list: reversion row unsat")        \
  X(EV_ST_AL_REV_AMBIG, ZKE_AMBIG, "add_account_storage_to_access_list: reversion row ambiguous")    \
  X(EV_ST_AL_PREV_TYPE, ZKE_ASSERT, "instruction.py:1086 value_prev.value() of a Word")              \
  X(EV_ST_REFUND_UNSAT, ZKE_UNSAT, "storage.py:82 tx_refund_write unsat")                            \
  X(EV_ST_REFUND_AMBIG, ZKE_AMBIG, "storage.py:82 tx_refund_write ambiguous")                        \
  X(EV_ST_REFUND_REV_UNSAT, ZKE_UNSAT, "storage.py:82 tx_refund_write: reversion row unsat")         \
  X(EV_ST_REFUND_REV_AMBIG, ZKE_AMBIG, "storage.py:82 tx_refund_write: reversion row ambiguous")     \
  X(EV_ST_REFUND_TYPE, ZKE_ASSERT, "instruction.py:950 value.value() of a Word")                     \
  X(EV_ST_REFUND_PREV_TYPE, ZKE_ASSERT, "instruction.py:950 value_prev.value() of a Word")           \
  X(EV_ST_REFUND_EQ, ZKE_ASSERT, "storage.py:125 gas_refund == the EIP-3529 rule")                   \
  X(EV_ST_WARM_BOOL, ZKE_ASSERT, "storage.py:39,136 select(is_warm, ..): not a bool")                \
  X(EV_CDL_OPCODE, ZKE_ASSERT, "calldataload.py:10 opcode == CALLDATALOAD")                          \
  X(EV_CDL_POP_UNSAT, ZKE_UNSAT, "calldataload.py:13 stack_pop unsat")                               \
  X(EV_CDL_POP_AMBIG, ZKE_AMBIG, "calldataload.py:13 stack_pop ambiguous")                           \
  X(EV_CDL_OFF_DOMAIN, ZKE_VALUE, "calldataload.py:13 word_to_fq: a half >= 2^128 -> OverflowError") \
  X(EV_CDL_OFF_RANGE, ZKE_RANGE, "calldataload.py:13 word_to_fq(.., 8): more than 8 bytes")          \
  X(EV_CDL_CC0_UNSAT, ZKE_UNSAT, "calldataload.py:16,20 call_context_lookup(TxId / CallerId) unsat") \
  X(EV_CDL_CC0_AMBIG, ZKE_AMBIG, "calldataload.py:16,20 call_context_lookup(TxId / CallerId) ambiguous") \
  X(EV_CDL_CC0_TYPE, ZKE_ASSERT, "calldataload.py:16,20 call_context_lookup(TxId / CallerId): .value() of a Word") \
  X(EV_CDL_CC1_UNSAT, ZKE_UNSAT, "calldataload.py:17,21 call_context_lookup(CallDataLength) unsat")  \
  X(EV_CDL_CC1_AMBIG, ZKE_AMBIG, "calldataload.py:17,21 call_context_lookup(CallDataLength) ambiguous") \
  X(EV_CDL_CC1_TYPE, ZKE_ASSERT, "calldataload.py:17,21 call_context_lookup(CallDataLength): .value() of a Word") \
  X(EV_CDL_CC2_UNSAT, ZKE_UNSAT, "calldataload.py:22 call_context_lookup(CallDataOffset) unsat")     \
  X(EV_CDL_CC2_AMBIG, ZKE_AMBIG, "calldataload.py:22 call_context_lookup(CallDataOffset) ambiguous") \
  X(EV_CDL_CC2_TYPE, ZKE_ASSERT, "calldataload.py:22 call_context_lookup(CallDataOffset): .value() of a Word") \
  X(EV_CDL_END_RANGE, ZKE_ASSERT, "memory_gadget.py:17 min(): addr_end exceeds 5 bytes (instruction.py:449)") \
  X(EV_CDL_START_RANGE, ZKE_ASSERT, "memory_gadget.py:17 min(): addr_start exceeds 5 bytes (instruction.py:450)") \
  X(EV_CDL_BYTE_UNSAT, ZKE_UNSAT, "calldataload.py:35,39 tx_calldata_lookup / memory_lookup unsat")  \
  X(EV_CDL_BYTE_AMBIG, ZKE_AMBIG, "calldataload.py:35,39 tx_calldata_lookup / memory_lookup ambiguous") \
  X(EV_CDL_BYTE_TYPE, ZKE_ASSERT, "calldataload.py:35,39 tx_calldata_lookup / memory_lookup: .value() of a Word") \
  X(EV_CDL_BYTES_VALUE, ZKE_VALUE, "calldataload.py:46 bytes() of a value > 255 -> ValueError")      \
  X(EV_CDL_PUSH_UNSAT, ZKE_UNSAT, "calldataload.py:47 stack_push unsat")                             \
  X(EV_CDL_PUSH_AMBIG, ZKE_AMBIG, "calldataload.py:47 stack_push ambiguous")                         \
  X(EV_CDL_EQ, ZKE_ASSERT, "calldataload.py:45-48 the 32 bytes == pushed word")                 \
  X(EV_LOG_RANGE5, ZKE_UNSAT, "log.py:11 range_lookup(opcode - LOG0, 5)")                            \
  X(EV_LOG_POP0_UNSAT, ZKE_UNSAT, "log.py:14 stack_pop mstart unsat")                                \
  X(EV_LOG_POP0_AMBIG, ZKE_AMBIG, "log.py:14 stack_pop mstart ambiguous")                            \
  X(EV_LOG_START_DOMAIN, ZKE_VALUE, "log.py:14 word_to_fq: a half >= 2^128 -> OverflowError")        \
  X(EV_LOG_START_RANGE, ZKE_RANGE, "log.py:14 word_to_fq(.., 8): more than 8 bytes")                 \
  X(EV_LOG_POP1_UNSAT, ZKE_UNSAT, "log.py:15 stack_pop msize unsat")                                 \
  X(EV_LOG_POP1_AMBIG, ZKE_AMBIG, "log.py:15 stack_pop msize ambiguous")                             \
  X(EV_LOG_SIZE_DOMAIN, ZKE_VALUE, "log.py:15 word_to_fq: a half >= 2^128 -> OverflowError")         \
  X(EV_LOG_SIZE_RANGE, ZKE_RANGE, "log.py:15 word_to_fq(.., 8): more than 8 bytes")                  \
  X(EV_LOG_TXID_UNSAT, ZKE_UNSAT, "log.py:18 call_context_lookup(TxId) unsat")                       \
  X(EV_LOG_TXID_AMBIG, ZKE_AMBIG, "log.py:18 call_context_lookup(TxId) ambiguous")                   \
  X(EV_LOG_TXID_TYPE, ZKE_ASSERT, "log.py:18 call_context_lookup(TxId): .value() of a Word")         \
  X(EV_LOG_STATIC_UNSAT, ZKE_UNSAT, "log.py:20-22 call_context_lookup(IsStatic) unsat")              \
  X(EV_LOG_STATIC_AMBIG, ZKE_AMBIG, "log.py:20-22 call_context_lookup(IsStatic) ambiguous")          \
  X(EV_LOG_STATIC_TYPE, ZKE_ASSERT, "log.py:20-22 call_context_lookup(IsStatic): .value() of a Word") \
  X(EV_LOG_STATIC_NONZERO, ZKE_ASSERT, "log.py:20-22 IsStatic == 0")                                 \
  X(EV_LOG_CALLEE_UNSAT, ZKE_UNSAT, "log.py:27 call_context_lookup_word(CalleeAddress) unsat")       \
  X(EV_LOG_CALLEE_AMBIG, ZKE_AMBIG, "log.py:27 call_context_lookup_word(CalleeAddress) ambiguous")   \
  X(EV_LOG_PERSIST_UNSAT, ZKE_UNSAT, "log.py:28 call_context_lookup(IsPersistent) unsat")            \
  X(EV_LOG_PERSIST_AMBIG, ZKE_AMBIG, "log.py:28 call_context_lookup(IsPersistent) ambiguous")        \
  X(EV_LOG_PERSIST_TYPE, ZKE_ASSERT, "log.py:28 call_context_lookup(IsPersistent): .value() of a Word") \
  X(EV_LOG_ADDR_UNSAT, ZKE_UNSAT, "log.py:32-34 tx_log_lookup_word(Address) unsat")                  \
  X(EV_LOG_ADDR_AMBIG, ZKE_AMBIG, "log.py:32-34 tx_log_lookup_word(Address) ambiguous")              \
  X(EV_LOG_ADDR_EQ, ZKE_ASSERT, "log.py:30-35 callee address == the log's address")                  \
  X(EV_LOG_TOPIC_POP_UNSAT, ZKE_UNSAT, "log.py:43 stack_pop topic unsat")                            \
  X(EV_LOG_TOPIC_POP_AMBIG, ZKE_AMBIG, "log.py:43 stack_pop topic ambiguous")                        \
  X(EV_LOG_TOPIC_UNSAT, ZKE_UNSAT, "log.py:47-52 tx_log_lookup_word(Topic, i) unsat")                \
  X(EV_LOG_TOPIC_AMBIG, ZKE_AMBIG, "log.py:47-52 tx_log_lookup_word(Topic, i) ambiguous")            \
  X(EV_LOG_TOPIC_EQ, ZKE_ASSERT, "log.py:45-53 topic == the log's topic")                            \
  X(EV_LOG_COPY_UNSAT, ZKE_UNSAT, "log.py:65-76 copy_lookup(Memory -> TxLog) unsat")                 \
  X(EV_LOG_COPY_AMBIG, ZKE_AMBIG, "log.py:65-76 copy_lookup(Memory -> TxLog) ambiguous")             \
  X(EV_LOG_MEMSIZE_RANGE, ZKE_RANGE, "log.py:83 memory_expansion_dynamic_length: memory size beyond 4 bytes") \
  X(EV_LOG_MEM_MAX, ZKE_ASSERT, "log.py:83 max(): curr.memory_word_size beyond 4 bytes")             \
  X(EV_EWP_OPCODE, ZKE_ASSERT, "error_write_protection.py:42-55 opcode modifies state")              \
  X(EV_EWP_STATIC_UNSAT, ZKE_UNSAT, "error_write_protection.py:59 call_context_lookup(IsStatic) unsat") \
  X(EV_EWP_STATIC_AMBIG, ZKE_AMBIG, "error_write_protection.py:59 call_context_lookup(IsStatic) ambiguous") \
  X(EV_EWP_STATIC_TYPE, ZKE_ASSERT, "error_write_protection.py:59 call_context_lookup(IsStatic): .value() of a Word") \
  X(EV_EWP_NOT_STATIC, ZKE_ASSERT, "error_write_protection.py:60 IsStatic == 1")                     \
  X(EV_EWP_VALUE_UNSAT, ZKE_UNSAT, "error_write_protection.py:65 stack_lookup(Read, 2) unsat")       \
  X(EV_EWP_VALUE_AMBIG, ZKE_AMBIG, "error_write_protection.py:65 stack_lookup(Read, 2) ambiguous")   \
  X(EV_EWP_VALUE_ZERO, ZKE_ASSERT, "error_write_protection.py:66 CALL value != 0")                   \
  X(EV_BH_POP_UNSAT, ZKE_UNSAT, "blockhash.py:9 stack_pop unsat")                                    \
  X(EV_BH_POP_AMBIG, ZKE_AMBIG, "blockhash.py:9 stack_pop ambiguous")                                \
  X(EV_BH_NUM_DOMAIN, ZKE_VALUE, "blockhash.py:9 word_to_u64: a half >= 2^128 -> OverflowError")     \
  X(EV_BH_NUM_RANGE, ZKE_RANGE, "blockhash.py:9 word_to_u64: more than 8 bytes")                     \
  X(EV_BH_CUR_UNSAT, ZKE_UNSAT, "blockhash.py:11 block_context_lookup(Number) unsat")                \
  X(EV_BH_CUR_AMBIG, ZKE_AMBIG, "blockhash.py:11 block_context_lookup(Number) ambiguous")            \
  X(EV_BH_CUR_TYPE, ZKE_ASSERT, "blockhash.py:11 block_context_lookup(Number): .value() of a Word")  \
  X(EV_BH_PUSH_UNSAT, ZKE_UNSAT, "blockhash.py:13 stack_push unsat")                                 \
  X(EV_BH_PUSH_AMBIG, ZKE_AMBIG, "blockhash.py:13 stack_push ambiguous")                             \
  X(EV_BH_CMP1_RANGE, ZKE_ASSERT, "blockhash.py:16 compare(block_number, current, 8): range assert") \
  X(EV_BH_CMP2_RANGE, ZKE_ASSERT, "blockhash.py:17 compare(current, 256 + block_number, 2): range assert") \
  X(EV_BH_HASH_UNSAT, ZKE_UNSAT, "blockhash.py:21-24 block_context_lookup_word(HistoryHash, block_number) unsat") \
  X(EV_BH_HASH_AMBIG, ZKE_AMBIG, "blockhash.py:21-24 block_context_lookup_word(HistoryHash, block_number) ambiguous") \
  X(EV_BH_EQ, ZKE_ASSERT, "blockhash.py:29 pushed word == expected block hash")                 \
  X(EV_EXP_RW0_UNSAT, ZKE_UNSAT, "exp.py:8 stack_pop base unsat")                                    \
  X(EV_EXP_RW0_AMBIG, ZKE_AMBIG, "exp.py:8 stack_pop base ambiguous")                                \
  X(EV_EXP_RW1_UNSAT, ZKE_UNSAT, "exp.py:9 stack_pop exponent unsat")                                \
  X(EV_EXP_RW1_AMBIG, ZKE_AMBIG, "exp.py:9 stack_pop exponent ambiguous")                            \
  X(EV_EXP_RW2_UNSAT, ZKE_UNSAT, "exp.py:10 stack_push unsat")                                       \
  X(EV_EXP_RW2_AMBIG, ZKE_AMBIG, "exp.py:10 stack_push ambiguous")                                   \
  X(EV_EXP_ZERO_LO, ZKE_ASSERT, "exp.py:20 exponent == 0 => exponentiation lo == 1")                 \
  X(EV_EXP_ZERO_HI, ZKE_ASSERT, "exp.py:21 exponent == 0 => exponentiation hi == 0")                 \
  X(EV_EXP_ONE_LO, ZKE_ASSERT, "exp.py:23 exponent == 1 => exponentiation lo == base lo")            \
  X(EV_EXP_ONE_HI, ZKE_ASSERT, "exp.py:24 exponent == 1 => exponentiation hi == base hi")            \
  X(EV_EXP_BASE_TO64, ZKE_VALUE, "exp.py:26 base.to_64s(): a half >= 2^128 -> OverflowError")        \
  X(EV_EXP_FIRST_UNSAT, ZKE_UNSAT, "exp.py:31 exp_lookup(identifier, single_step, base limbs, exponent) unsat") \
  X(EV_EXP_FIRST_AMBIG, ZKE_AMBIG, "exp.py:31 exp_lookup(identifier, single_step, base limbs, exponent) ambiguous") \
  X(EV_EXP_LAST_UNSAT, ZKE_UNSAT, "exp.py:33 exp_lookup(identifier, 1, base limbs, 2) unsat")        \
  X(EV_EXP_LAST_AMBIG, ZKE_AMBIG, "exp.py:33 exp_lookup(identifier, 1, base limbs, 2) ambiguous")    \
  X(EV_EXP_CARRY_LO, ZKE_RANGE, "exp.py:36 mul_add_words(base, base, 0, base^2): range_check(carry_lo, 9)") \
  X(EV_EXP_CARRY_HI, ZKE_RANGE, "exp.py:36 mul_add_words: range_check(carry_hi, 9)")                 \
  X(EV_EXP_RESULT, ZKE_ASSERT, "exp.py:39 looked-up exponentiation == pushed word")                  \
  X(EV_EXP_EXPONENT_BYTES, ZKE_VALUE, "exp.py:41 byte_size(exponent): to_le_bytes of a half >= 2^128 -> OverflowError")                 \
  X(EV_ECS_OPCODE, ZKE_ASSERT, "error_code_store.py:20 / error_invalid_creation_code.py:15 opcode == RETURN") \
  X(EV_ECS_IS_CREATE, ZKE_ASSERT, "error_code_store.py:23 / error_invalid_creation_code.py:18 is_create == 1") \
  X(EV_ECS_LEN_UNSAT, ZKE_UNSAT, "error_code_store.py:26 stack_lookup(Read, 1) / error_invalid_creation_code.py:21 stack_pop unsat") \
  X(EV_ECS_LEN_AMBIG, ZKE_AMBIG, "error_code_store.py:26 stack_lookup(Read, 1) / error_invalid_creation_code.py:21 stack_pop ambiguous") \
  X(EV_ECS_LEN_DOMAIN, ZKE_VALUE, "word_to_fq: a half >= 2^128 -> OverflowError")                    \
  X(EV_ECS_LEN_RANGE, ZKE_RANGE, "word_to_fq(.., 5): more than 5 bytes")                             \
  X(EV_ECS_STATIC_UNSAT, ZKE_UNSAT, "error_code_store.py:30 call_context_lookup(IsStatic) unsat")    \
  X(EV_ECS_STATIC_AMBIG, ZKE_AMBIG, "error_code_store.py:30 call_context_lookup(IsStatic) ambiguous") \
  X(EV_ECS_STATIC_TYPE, ZKE_ASSERT, "error_code_store.py:30 call_context_lookup(IsStatic): .value() of a Word") \
  X(EV_ECS_STATIC_NONZERO, ZKE_ASSERT, "error_code_store.py:31 IsStatic == 0")                       \
  X(EV_ECS_SIZE_RANGE, ZKE_ASSERT, "error_code_store.py:34 compare(MAX_CODE_SIZE, return_length, 2): range assert") \
  X(EV_ECS_GAS_RANGE, ZKE_ASSERT, "error_code_store.py:38-40 compare(gas_left, deposit cost, 8): range assert") \
  X(EV_ECS_NEITHER, ZKE_ASSERT, "error_code_store.py:43 neither out of gas nor over the maximum code size") \
  X(EV_ECS_BYTE_UNSAT, ZKE_UNSAT, "error_invalid_creation_code.py:24 memory_lookup(Read, return_offset) unsat") \
  X(EV_ECS_BYTE_AMBIG, ZKE_AMBIG, "error_invalid_creation_code.py:24 memory_lookup(Read, return_offset) ambiguous") \
  X(EV_ECS_BYTE_TYPE, ZKE_ASSERT, "error_invalid_creation_code.py:24 memory_lookup(Read, return_offset): .value() of a Word") \
  X(EV_ECS_FIRST_BYTE, ZKE_ASSERT, "error_invalid_creation_code.py:27 first byte == 0xEF")                 \
  X(EV_RET_SUCCESS_UNSAT, ZKE_UNSAT, "return_revert.py:17 call_context_lookup(IsSuccess) unsat")     \
  X(EV_RET_SUCCESS_AMBIG, ZKE_AMBIG, "return_revert.py:17 call_context_lookup(IsSuccess) ambiguous") \
  X(EV_RET_SUCCESS_TYPE, ZKE_ASSERT, "return_revert.py:17 call_context_lookup(IsSuccess): .value() of a Word") \
  X(EV_RET_SUCCESS_EQ, ZKE_ASSERT, "return_revert.py:18 is_success == is_return")                    \
  X(EV_RET_POP0_UNSAT, ZKE_UNSAT, "return_revert.py:20 stack_pop return offset unsat")               \
  X(EV_RET_POP0_AMBIG, ZKE_AMBIG, "return_revert.py:20 stack_pop return offset ambiguous")           \
  X(EV_RET_POP1_UNSAT, ZKE_UNSAT, "return_revert.py:21 stack_pop return length unsat")               \
  X(EV_RET_POP1_AMBIG, ZKE_AMBIG, "return_revert.py:21 stack_pop return length ambiguous")           \
  X(EV_RET_OFF_DOMAIN, ZKE_VALUE, "return_revert.py:23 word_to_fq: a half >= 2^128 -> OverflowError") \
  X(EV_RET_OFF_RANGE, ZKE_RANGE, "return_revert.py:23 word_to_fq(.., 5): more than 5 bytes")         \
  X(EV_RET_LEN_DOMAIN, ZKE_VALUE, "return_revert.py:24 word_to_fq: a half >= 2^128 -> OverflowError") \
  X(EV_RET_LEN_RANGE, ZKE_RANGE, "return_revert.py:24 word_to_fq(.., 5): more than 5 bytes")         \
  X(EV_RET_CALLEE_UNSAT, ZKE_UNSAT, "return_revert.py:33-35 call_context_lookup_word(CalleeAddress) unsat") \
  X(EV_RET_CALLEE_AMBIG, ZKE_AMBIG, "return_revert.py:33-35 call_context_lookup_word(CalleeAddress) ambiguous") \
  X(EV_RET_CALLEE_DOMAIN, ZKE_VALUE, "return_revert.py:36 word_to_address: a half >= 2^128 -> OverflowError") \
  X(EV_RET_CALLEE_RANGE, ZKE_RANGE, "return_revert.py:36 word_to_address: more than 20 bytes")       \
  X(EV_RET_HASH_WRITE_UNSAT, ZKE_UNSAT, "return_revert.py:37-39 account_write_word(CodeHash) unsat") \
  X(EV_RET_HASH_WRITE_AMBIG, ZKE_AMBIG, "return_revert.py:37-39 account_write_word(CodeHash) ambiguous") \
  X(EV_RET_HASH_PREV, ZKE_ASSERT, "return_revert.py:40 previous code hash == EMPTY_HASH")            \
  X(EV_RET_HASH_CUR, ZKE_ASSERT, "return_revert.py:41 written code hash == curr.code_hash")          \
  X(EV_RET_MAX_CODE_SIZE, ZKE_UNSAT, "return_revert.py:44 range_lookup(return_length, MAX_CODE_SIZE)") \
  X(EV_RET_COPY_CODE_UNSAT, ZKE_UNSAT, "return_revert.py:54-64 copy_lookup(Memory -> Bytecode) unsat") \
  X(EV_RET_COPY_CODE_AMBIG, ZKE_AMBIG, "return_revert.py:54-64 copy_lookup(Memory -> Bytecode) ambiguous") \
  X(EV_RET_COPY_CODE_INC, ZKE_ASSERT, "return_revert.py:65 copy_rwc_inc == copy_length")             \
  X(EV_RET_CODE_LEN_UNSAT, ZKE_UNSAT, "return_revert.py:68 bytecode_length(code_hash) unsat")        \
  X(EV_RET_CODE_LEN_AMBIG, ZKE_AMBIG, "return_revert.py:68 bytecode_length(code_hash) ambiguous")    \
  X(EV_RET_CODE_LEN_EQ, ZKE_ASSERT, "return_revert.py:69 code size == copy_length")                  \
  X(EV_RET_RDO_UNSAT, ZKE_UNSAT, "return_revert.py:76-78 call_context_lookup(ReturnDataOffset) unsat") \
  X(EV_RET_RDO_AMBIG, ZKE_AMBIG, "return_revert.py:76-78 call_context_lookup(ReturnDataOffset) ambiguous") \
  X(EV_RET_RDO_TYPE, ZKE_ASSERT, "return_revert.py:76-78 call_context_lookup(ReturnDataOffset): .value() of a Word") \
  X(EV_RET_RDL_UNSAT, ZKE_UNSAT, "return_revert.py:79-81 call_context_lookup(ReturnDataLength) unsat") \
  X(EV_RET_RDL_AMBIG, ZKE_AMBIG, "return_revert.py:79-81 call_context_lookup(ReturnDataLength) ambiguous") \
  X(EV_RET_RDL_TYPE, ZKE_ASSERT, "return_revert.py:79-81 call_context_lookup(ReturnDataLength): .value() of a Word") \
  X(EV_RET_MIN_RANGE, ZKE_ASSERT, "return_revert.py:82 min(): caller return length exceeds 5 bytes") \
  X(EV_RET_COPY_UNSAT, ZKE_UNSAT, "return_revert.py:83-93 copy_lookup(Memory -> caller Memory) unsat") \
  X(EV_RET_COPY_AMBIG, ZKE_AMBIG, "return_revert.py:83-93 copy_lookup(Memory -> caller Memory) ambiguous") \
  X(EV_RET_COPY_INC, ZKE_ASSERT, "return_revert.py:94 copy_rwc_inc == 2 * copy_length")              \
  X(EV_RET_ROOT_ENDTX, ZKE_ASSERT, "return_revert.py:101 is_root == (next state is EndTx)")          \
  X(EV_RET_MEMSIZE_RANGE, ZKE_RANGE, "return_revert.py:103 memory_expansion_dynamic_length: memory size beyond 4 bytes") \
  X(EV_RET_MEM_MAX, ZKE_ASSERT, "return_revert.py:103 max(): curr.memory_word_size beyond 4 bytes")  \
  X(EV_RET_PERSIST_UNSAT, ZKE_UNSAT, "return_revert.py:115-117 call_context_lookup(IsPersistent) unsat") \
  X(EV_RET_PERSIST_AMBIG, ZKE_AMBIG, "return_revert.py:115-117 call_context_lookup(IsPersistent) ambiguous") \
  X(EV_RET_PERSIST_TYPE, ZKE_ASSERT, "return_revert.py:115-117 call_context_lookup(IsPersistent): .value() of a Word") \
  X(EV_RET_PERSIST_EQ, ZKE_ASSERT, "return_revert.py:118 is_persistent == is_return")                \
  X(EV_RET_RWC, ZKE_ASSERT, "return_revert.py:121-125 rw_counter delta")                             \
  X(EV_RET_GAS, ZKE_ASSERT, "return_revert.py:121-125 gas_left to callee gas left")                  \
  X(EV_RET_CALL_ID, ZKE_ASSERT, "return_revert.py:121-125 call_id same")                 \
  X(EV_EOC_OPCODE, ZKE_ASSERT, "error_oog_call.py:19 opcode is CALL / CALLCODE / DELEGATECALL / STATICCALL") \
  X(EV_EOC_TXID_UNSAT, ZKE_UNSAT, "error_oog_call.py:21 call_context_lookup(TxId) unsat")            \
  X(EV_EOC_TXID_AMBIG, ZKE_AMBIG, "error_oog_call.py:21 call_context_lookup(TxId) ambiguous")        \
  X(EV_EOC_TXID_TYPE, ZKE_ASSERT, "error_oog_call.py:21 call_context_lookup(TxId): .value() of a Word") \
  X(EV_EOC_POP0_UNSAT, ZKE_UNSAT, "call_gadget.py:53-63 stack_pop gas unsat")                        \
  X(EV_EOC_POP0_AMBIG, ZKE_AMBIG, "call_gadget.py:53-63 stack_pop gas ambiguous")                    \
  X(EV_EOC_POP1_UNSAT, ZKE_UNSAT, "call_gadget.py:53-63 stack_pop callee address unsat")             \
  X(EV_EOC_POP1_AMBIG, ZKE_AMBIG, "call_gadget.py:53-63 stack_pop callee address ambiguous")         \
  X(EV_EOC_POP2_UNSAT, ZKE_UNSAT, "call_gadget.py:53-63 stack_pop value unsat")                      \
  X(EV_EOC_POP2_AMBIG, ZKE_AMBIG, "call_gadget.py:53-63 stack_pop value ambiguous")                  \
  X(EV_EOC_POP3_UNSAT, ZKE_UNSAT, "call_gadget.py:53-63 stack_pop cd_offset unsat")                  \
  X(EV_EOC_POP3_AMBIG, ZKE_AMBIG, "call_gadget.py:53-63 stack_pop cd_offset ambiguous")              \
  X(EV_EOC_POP4_UNSAT, ZKE_UNSAT, "call_gadget.py:53-63 stack_pop cd_length unsat")                  \
  X(EV_EOC_POP4_AMBIG, ZKE_AMBIG, "call_gadget.py:53-63 stack_pop cd_length ambiguous")              \
  X(EV_EOC_POP5_UNSAT, ZKE_UNSAT, "call_gadget.py:53-63 stack_pop rd_offset unsat")                  \
  X(EV_EOC_POP5_AMBIG, ZKE_AMBIG, "call_gadget.py:53-63 stack_pop rd_offset ambiguous")              \
  X(EV_EOC_POP6_UNSAT, ZKE_UNSAT, "call_gadget.py:53-63 stack_pop rd_length unsat")                  \
  X(EV_EOC_POP6_AMBIG, ZKE_AMBIG, "call_gadget.py:53-63 stack_pop rd_length ambiguous")              \
  X(EV_EOC_PUSH_UNSAT, ZKE_UNSAT, "call_gadget.py:64 stack_push result unsat")                       \
  X(EV_EOC_PUSH_AMBIG, ZKE_AMBIG, "call_gadget.py:64 stack_push result ambiguous")                   \
  X(EV_EOC_RESULT_WORD, ZKE_ASSERT, "call_gadget.py:66 result == Word.from_lo(is_success)")          \
  X(EV_EOC_RESULT_BOOL, ZKE_ASSERT, "call_gadget.py:69 is_success is a bool")                        \
  X(EV_EOC_RESULT_ZERO, ZKE_ASSERT, "call_gadget.py:71 is_success == 0 (failed call)")               \
  X(EV_EOC_GAS_DOMAIN, ZKE_VALUE, "call_gadget.py:73 gas: word_to_fq of a half >= 2^128 -> OverflowError") \
  X(EV_EOC_GAS_RANGE, ZKE_RANGE, "call_gadget.py:73 gas: more than 8 bytes")                         \
  X(EV_EOC_CALLEE_DOMAIN, ZKE_VALUE, "call_gadget.py:85 callee address: word_to_fq of a half >= 2^128 -> OverflowError") \
  X(EV_EOC_CALLEE_RANGE, ZKE_RANGE, "call_gadget.py:85 callee address: more than 20 bytes")          \
  X(EV_EOC_CDLEN_DOMAIN, ZKE_VALUE, "call_gadget.py:86 cd_length: word_to_fq of a half >= 2^128 -> OverflowError") \
  X(EV_EOC_CDLEN_RANGE, ZKE_RANGE, "call_gadget.py:86 cd_length: more than 5 bytes")                 \
  X(EV_EOC_CDOFF_DOMAIN, ZKE_VALUE, "call_gadget.py:86 cd_offset: word_to_fq of a half >= 2^128 -> OverflowError") \
  X(EV_EOC_CDOFF_RANGE, ZKE_RANGE, "call_gadget.py:86 cd_offset: more than 5 bytes")                 \
  X(EV_EOC_RDLEN_DOMAIN, ZKE_VALUE, "call_gadget.py:87 rd_length: word_to_fq of a half >= 2^128 -> OverflowError") \
  X(EV_EOC_RDLEN_RANGE, ZKE_RANGE, "call_gadget.py:87 rd_length: more than 5 bytes")                 \
  X(EV_EOC_RDOFF_DOMAIN, ZKE_VALUE, "call_gadget.py:87 rd_offset: word_to_fq of a half >= 2^128 -> OverflowError") \
  X(EV_EOC_RDOFF_RANGE, ZKE_RANGE, "call_gadget.py:87 rd_offset: more than 5 bytes")                 \
  X(EV_EOC_CD_MEMSIZE_RANGE, ZKE_RANGE, "call_gadget.py:92 memory_expansion_dynamic_length: call-data memory size beyond 4 bytes") \
  X(EV_EOC_MEM_MAX, ZKE_ASSERT, "call_gadget.py:92 max(): curr.memory_word_size beyond 4 bytes")     \
  X(EV_EOC_RD_MEMSIZE_RANGE, ZKE_RANGE, "call_gadget.py:92 memory_expansion_dynamic_length: return-data memory size beyond 4 bytes") \
  X(EV_EOC_HASH_UNSAT, ZKE_UNSAT, "call_gadget.py:100 account_read_word(CodeHash) unsat")            \
  X(EV_EOC_HASH_AMBIG, ZKE_AMBIG, "call_gadget.py:100 account_read_word(CodeHash) ambiguous")        \
  X(EV_EOC_AL_UNSAT, ZKE_UNSAT, "error_oog_call.py:29 read_account_to_access_list unsat")            \
  X(EV_EOC_AL_AMBIG, ZKE_AMBIG, "error_oog_call.py:29 read_account_to_access_list ambiguous")        \
  X(EV_EOC_AL_PREV_TYPE, ZKE_ASSERT, "instruction.py:1069 value_prev.value() of a Word")             \
  X(EV_EOC_WARM_BOOL, ZKE_ASSERT, "call_gadget.py:114 select(is_warm_access, ..): not a bool")       \
  X(EV_EOC_CMP_RANGE, ZKE_ASSERT, "error_oog_call.py:35 compare(gas_left, gas_cost, 8): range assert") \
  X(EV_EOC_NOT_ENOUGH, ZKE_ASSERT, "error_oog_call.py:36 gas_left < gas_cost")                 \
  X(EV_CALL_RESP_OPCODE, ZKE_UNSAT, "callop.py:17 responsible_opcode_lookup(opcode)")                \
  X(EV_CALL_TXID_UNSAT, ZKE_UNSAT, "callop.py:21 call_context_lookup(TxId) unsat")                   \
  X(EV_CALL_TXID_AMBIG, ZKE_AMBIG, "callop.py:21 call_context_lookup(TxId) ambiguous")               \
  X(EV_CALL_TXID_TYPE, ZKE_ASSERT, "callop.py:21 call_context_lookup(TxId): .value() of a Word")     \
  X(EV_CALL_REVEND_UNSAT, ZKE_UNSAT, "callop.py:22 reversion_info: RwCounterEndOfReversion unsat")   \
  X(EV_CALL_REVEND_AMBIG, ZKE_AMBIG, "callop.py:22 reversion_info: RwCounterEndOfReversion ambiguous") \
  X(EV_CALL_REVEND_TYPE, ZKE_ASSERT, "callop.py:22 reversion_info: RwCounterEndOfReversion: .value() of a Word") \
  X(EV_CALL_PERSIST_UNSAT, ZKE_UNSAT, "callop.py:22 reversion_info: IsPersistent unsat")             \
  X(EV_CALL_PERSIST_AMBIG, ZKE_AMBIG, "callop.py:22 reversion_info: IsPersistent ambiguous")         \
  X(EV_CALL_PERSIST_TYPE, ZKE_ASSERT, "callop.py:22 reversion_info: IsPersistent: .value() of a Word") \
  X(EV_CALL_SELF_UNSAT, ZKE_UNSAT, "callop.py:23-25 call_context_lookup_word(CalleeAddress) unsat")  \
  X(EV_CALL_SELF_AMBIG, ZKE_AMBIG, "callop.py:23-25 call_context_lookup_word(CalleeAddress) ambiguous") \
  X(EV_CALL_SELF_DOMAIN, ZKE_VALUE, "callop.py:26 word_to_address(current callee address): word_to_fq of a half >= 2^128 -> OverflowError") \
  X(EV_CALL_SELF_RANGE, ZKE_RANGE, "callop.py:26 word_to_address(current callee address): more than 20 bytes") \
  X(EV_CALL_STATIC_UNSAT, ZKE_UNSAT, "callop.py:27 call_context_lookup(IsStatic) unsat")             \
  X(EV_CALL_STATIC_AMBIG, ZKE_AMBIG, "callop.py:27 call_context_lookup(IsStatic) ambiguous")         \
  X(EV_CALL_STATIC_TYPE, ZKE_ASSERT, "callop.py:27 call_context_lookup(IsStatic): .value() of a Word") \
  X(EV_CALL_DEPTH_UNSAT, ZKE_UNSAT, "callop.py:28 call_context_lookup(Depth) unsat")                 \
  X(EV_CALL_DEPTH_AMBIG, ZKE_AMBIG, "callop.py:28 call_context_lookup(Depth) ambiguous")             \
  X(EV_CALL_DEPTH_TYPE, ZKE_ASSERT, "callop.py:28 call_context_lookup(Depth): .value() of a Word")   \
  X(EV_CALL_PCALLER_UNSAT, ZKE_UNSAT, "callop.py:31 call_context_lookup_word(CallerAddress) (DELEGATECALL) unsat") \
  X(EV_CALL_PCALLER_AMBIG, ZKE_AMBIG, "callop.py:31 call_context_lookup_word(CallerAddress) (DELEGATECALL) ambiguous") \
  X(EV_CALL_PVALUE_UNSAT, ZKE_UNSAT, "callop.py:32 call_context_lookup_word(Value) (DELEGATECALL) unsat") \
  X(EV_CALL_PVALUE_AMBIG, ZKE_AMBIG, "callop.py:32 call_context_lookup_word(Value) (DELEGATECALL) ambiguous") \
  X(EV_CALL_OPCODE, ZKE_ASSERT, "call_gadget.py:51 exactly one of CALL / CALLCODE / DELEGATECALL / STATICCALL") \
  X(EV_CALL_POP0_UNSAT, ZKE_UNSAT, "call_gadget.py:53-63 stack_pop gas unsat")                       \
  X(EV_CALL_POP0_AMBIG, ZKE_AMBIG, "call_gadget.py:53-63 stack_pop gas ambiguous")                   \
  X(EV_CALL_POP1_UNSAT, ZKE_UNSAT, "call_gadget.py:53-63 stack_pop callee address unsat")            \
  X(EV_CALL_POP1_AMBIG, ZKE_AMBIG, "call_gadget.py:53-63 stack_pop callee address ambiguous")        \
  X(EV_CALL_POP2_UNSAT, ZKE_UNSAT, "call_gadget.py:53-63 stack_pop value unsat")                     \
  X(EV_CALL_POP2_AMBIG, ZKE_AMBIG, "call_gadget.py:53-63 stack_pop value ambiguous")                 \
  X(EV_CALL_POP3_UNSAT, ZKE_UNSAT, "call_gadget.py:53-63 stack_pop cd_offset unsat")                 \
  X(EV_CALL_POP3_AMBIG, ZKE_AMBIG, "call_gadget.py:53-63 stack_pop cd_offset ambiguous")             \
  X(EV_CALL_POP4_UNSAT, ZKE_UNSAT, "call_gadget.py:53-63 stack_pop cd_length unsat")                 \
  X(EV_CALL_POP4_AMBIG, ZKE_AMBIG, "call_gadget.py:53-63 stack_pop cd_length ambiguous")             \
  X(EV_CALL_POP5_UNSAT, ZKE_UNSAT, "call_gadget.py:53-63 stack_pop rd_offset unsat")                 \
  X(EV_CALL_POP5_AMBIG, ZKE_AMBIG, "call_gadget.py:53-63 stack_pop rd_offset ambiguous")             \
  X(EV_CALL_POP6_UNSAT, ZKE_UNSAT, "call_gadget.py:53-63 stack_pop rd_length unsat")                 \
  X(EV_CALL_POP6_AMBIG, ZKE_AMBIG, "call_gadget.py:53-63 stack_pop rd_length ambiguous")             \
  X(EV_CALL_PUSH_UNSAT, ZKE_UNSAT, "call_gadget.py:64 stack_push result unsat")                      \
  X(EV_CALL_PUSH_AMBIG, ZKE_AMBIG, "call_gadget.py:64 stack_push result ambiguous")                  \
  X(EV_CALL_RESULT_WORD, ZKE_ASSERT, "call_gadget.py:66 result == Word.from_lo(is_success)")         \
  X(EV_CALL_RESULT_BOOL, ZKE_ASSERT, "call_gadget.py:69 is_success is a bool")                       \
  X(EV_CALL_GAS_DOMAIN, ZKE_VALUE, "call_gadget.py:73 gas: word_to_fq of a half >= 2^128 -> OverflowError") \
  X(EV_CALL_GAS_RANGE, ZKE_RANGE, "call_gadget.py:73 gas: more than 8 bytes")                        \
  X(EV_CALL_CALLEE_DOMAIN, ZKE_VALUE, "call_gadget.py:85 callee address: word_to_fq of a half >= 2^128 -> OverflowError") \
  X(EV_CALL_CALLEE_RANGE, ZKE_RANGE, "call_gadget.py:85 callee address: more than 20 bytes")         \
  X(EV_CALL_CDLEN_DOMAIN, ZKE_VALUE, "call_gadget.py:86 cd_length: word_to_fq of a half >= 2^128 -> OverflowError") \
  X(EV_CALL_CDLEN_RANGE, ZKE_RANGE, "call_gadget.py:86 cd_length: more than 5 bytes")                \
  X(EV_CALL_CDOFF_DOMAIN, ZKE_VALUE, "call_gadget.py:86 cd_offset: word_to_fq of a half >= 2^128 -> OverflowError") \
  X(EV_CALL_CDOFF_RANGE, ZKE_RANGE, "call_gadget.py:86 cd_offset: more than 5 bytes")                \
  X(EV_CALL_RDLEN_DOMAIN, ZKE_VALUE, "call_gadget.py:87 rd_length: word_to_fq of a half >= 2^128 -> OverflowError") \
  X(EV_CALL_RDLEN_RANGE, ZKE_RANGE, "call_gadget.py:87 rd_length: more than 5 bytes")                \
  X(EV_CALL_RDOFF_DOMAIN, ZKE_VALUE, "call_gadget.py:87 rd_offset: word_to_fq of a half >= 2^128 -> OverflowError") \
  X(EV_CALL_RDOFF_RANGE, ZKE_RANGE, "call_gadget.py:87 rd_offset: more than 5 bytes")                \
  X(EV_CALL_CD_MEMSIZE_RANGE, ZKE_RANGE, "call_gadget.py:92 memory_expansion_dynamic_length: call-data memory size beyond 4 bytes") \
  X(EV_CALL_MEM_MAX, ZKE_ASSERT, "call_gadget.py:92 max(): curr.memory_word_size beyond 4 bytes")    \
  X(EV_CALL_RD_MEMSIZE_RANGE, ZKE_RANGE, "call_gadget.py:92 memory_expansion_dynamic_length: return-data memory size beyond 4 bytes") \
  X(EV_CALL_HASH_UNSAT, ZKE_UNSAT, "call_gadget.py:100 account_read_word(CodeHash) unsat")           \
  X(EV_CALL_HASH_AMBIG, ZKE_AMBIG, "call_gadget.py:100 account_read_word(CodeHash) ambiguous")       \
  X(EV_CALL_CALLER_WORD, ZKE_ASSERT, "callop.py:51-53 select_word: a half of the parent caller address >= 2^128") \
  X(EV_CALL_CALLER_DOMAIN, ZKE_VALUE, "callop.py:54 word_to_address(caller address): word_to_fq of a half >= 2^128 -> OverflowError") \
  X(EV_CALL_CALLER_RANGE, ZKE_RANGE, "callop.py:54 word_to_address(caller address): more than 20 bytes") \
  X(EV_CALL_AL_UNSAT, ZKE_UNSAT, "callop.py:57-59 add_account_to_access_list unsat")                 \
  X(EV_CALL_AL_AMBIG, ZKE_AMBIG, "callop.py:57-59 add_account_to_access_list ambiguous")             \
  X(EV_CALL_AL_REV_UNSAT, ZKE_UNSAT, "callop.py:57-59 add_account_to_access_list: reversion row unsat") \
  X(EV_CALL_AL_REV_AMBIG, ZKE_AMBIG, "callop.py:57-59 add_account_to_access_list: reversion row ambiguous") \
  X(EV_CALL_AL_PREV_TYPE, ZKE_ASSERT, "instruction.py:1057 value_prev.value() of a Word")            \
  X(EV_CALL_VALUE_STATIC, ZKE_ASSERT, "callop.py:63 has_value * is_static == 0")                     \
  X(EV_CALL_CREVEND_UNSAT, ZKE_UNSAT, "callop.py:66 reversion_info(callee): RwCounterEndOfReversion unsat") \
  X(EV_CALL_CREVEND_AMBIG, ZKE_AMBIG, "callop.py:66 reversion_info(callee): RwCounterEndOfReversion ambiguous") \
  X(EV_CALL_CREVEND_TYPE, ZKE_ASSERT, "callop.py:66 reversion_info(callee): RwCounterEndOfReversion: .value() of a Word") \
  X(EV_CALL_CPERSIST_UNSAT, ZKE_UNSAT, "callop.py:66 reversion_info(callee): IsPersistent unsat")    \
  X(EV_CALL_CPERSIST_AMBIG, ZKE_AMBIG, "callop.py:66 reversion_info(callee): IsPersistent ambiguous") \
  X(EV_CALL_CPERSIST_TYPE, ZKE_ASSERT, "callop.py:66 reversion_info(callee): IsPersistent: .value() of a Word") \
  X(EV_CALL_CPERSIST_EQ, ZKE_ASSERT, "callop.py:67-70 callee is_persistent == caller is_persistent * is_success") \
  X(EV_CALL_CREVEND_EQ, ZKE_ASSERT, "callop.py:76-79 callee rw_counter_end_of_reversion == caller rw_counter_of_reversion()") \
  X(EV_CALL_BAL_UNSAT, ZKE_UNSAT, "callop.py:84 account_read_word(caller, Balance) unsat")           \
  X(EV_CALL_BAL_AMBIG, ZKE_AMBIG, "callop.py:84 account_read_word(caller, Balance) ambiguous")       \
  X(EV_CALL_BAL_CMP_RANGE, ZKE_ASSERT, "callop.py:86 compare_word(caller_balance, value): 16-byte range assert") \
  X(EV_CALL_DEPTH_RANGE, ZKE_ASSERT, "callop.py:87 compare(depth, 1025, 2): range assert")           \
  X(EV_CALL_PRECHECK_SUCCESS, ZKE_ASSERT, "callop.py:91-92 pre-check failed => is_success == 0")     \
  X(EV_CALL_SEND_UNSAT, ZKE_UNSAT, "callop.py:96 transfer: sub_balance account write unsat")         \
  X(EV_CALL_SEND_AMBIG, ZKE_AMBIG, "callop.py:96 transfer: sub_balance account write ambiguous")     \
  X(EV_CALL_SEND_REV_UNSAT, ZKE_UNSAT, "callop.py:96 transfer: sub_balance reversion row unsat")     \
  X(EV_CALL_SEND_REV_AMBIG, ZKE_AMBIG, "callop.py:96 transfer: sub_balance reversion row ambiguous") \
  X(EV_CALL_SEND_EQ, ZKE_ASSERT, "instruction.py:1011 sender balance_prev == balance + value")       \
  X(EV_CALL_SEND_CARRY, ZKE_ASSERT, "instruction.py:1012 sender carry == 0")                         \
  X(EV_CALL_RECV_UNSAT, ZKE_UNSAT, "callop.py:96 transfer: add_balance account write unsat")         \
  X(EV_CALL_RECV_AMBIG, ZKE_AMBIG, "callop.py:96 transfer: add_balance account write ambiguous")     \
  X(EV_CALL_RECV_REV_UNSAT, ZKE_UNSAT, "callop.py:96 transfer: add_balance reversion row unsat")     \
  X(EV_CALL_RECV_REV_AMBIG, ZKE_AMBIG, "callop.py:96 transfer: add_balance reversion row ambiguous") \
  X(EV_CALL_RECV_EQ, ZKE_ASSERT, "instruction.py:997 receiver balance == balance_prev + value")      \
  X(EV_CALL_RECV_CARRY, ZKE_ASSERT, "instruction.py:998 receiver carry == 0")                        \
  X(EV_CALL_CALLCODE_BALANCE, ZKE_ASSERT, "callop.py:98-99 CALLCODE succeeded => balance sufficient") \
  X(EV_CALL_WARM_BOOL, ZKE_ASSERT, "call_gadget.py:114 select(is_warm_access, ..): not a bool")      \
  X(EV_CALL_GAS_64TH_RANGE, ZKE_RANGE, "callop.py:110 constant_divmod(gas_available, 64, 8): quotient beyond 8 bytes (not enough gas)") \
  X(EV_CALL_GAS_MIN_RANGE, ZKE_ASSERT, "callop.py:114 min(all_but_one_64th_gas, gas, 8): range assert") \
  X(EV_CALL_PRECOMPILE_STATE, ZKE_ASSERT, "callop.py:121-123 callee is a precompile <=> the next state is a precompile state") \
  X(EV_CALL_LAST0_UNSAT, ZKE_UNSAT, "callop.py:130-138 call_context_lookup(LastCalleeId, Write) unsat") \
  X(EV_CALL_LAST0_AMBIG, ZKE_AMBIG, "callop.py:130-138 call_context_lookup(LastCalleeId, Write) ambiguous") \
  X(EV_CALL_LAST0_TYPE, ZKE_ASSERT, "callop.py:130-138 call_context_lookup(LastCalleeId, Write): .value() of a Word") \
  X(EV_CALL_LAST0_EQ, ZKE_ASSERT, "callop.py:135-138 LastCalleeId == 0")                             \
  X(EV_CALL_LAST1_UNSAT, ZKE_UNSAT, "callop.py:130-138 call_context_lookup(LastCalleeReturnDataOffset, Write) unsat") \
  X(EV_CALL_LAST1_AMBIG, ZKE_AMBIG, "callop.py:130-138 call_context_lookup(LastCalleeReturnDataOffset, Write) ambiguous") \
  X(EV_CALL_LAST1_TYPE, ZKE_ASSERT, "callop.py:130-138 call_context_lookup(LastCalleeReturnDataOffset, Write): .value() of a Word") \
  X(EV_CALL_LAST1_EQ, ZKE_ASSERT, "callop.py:135-138 LastCalleeReturnDataOffset == 0")               \
  X(EV_CALL_LAST2_UNSAT, ZKE_UNSAT, "callop.py:130-138 call_context_lookup(LastCalleeReturnDataLength, Write) unsat") \
  X(EV_CALL_LAST2_AMBIG, ZKE_AMBIG, "callop.py:130-138 call_context_lookup(LastCalleeReturnDataLength, Write) ambiguous") \
  X(EV_CALL_LAST2_TYPE, ZKE_ASSERT, "callop.py:130-138 call_context_lookup(LastCalleeReturnDataLength, Write): .value() of a Word") \
  X(EV_CALL_LAST2_EQ, ZKE_ASSERT, "callop.py:135-138 LastCalleeReturnDataLength == 0")               \
  X(EV_CALL_SAME_RWC, ZKE_ASSERT, "callop.py:140-151 stay in the caller: rw_counter delta")          \
  X(EV_CALL_SAME_PC, ZKE_ASSERT, "callop.py:140-151 stay in the caller: program_counter + 1")        \
  X(EV_CALL_SAME_SP, ZKE_ASSERT, "callop.py:140-151 stay in the caller: stack_pointer delta")        \
  X(EV_CALL_SAME_GAS, ZKE_ASSERT, "callop.py:140-151 stay in the caller: gas_left delta")            \
  X(EV_CALL_SAME_MEM, ZKE_ASSERT, "callop.py:140-151 stay in the caller: memory_word_size to next")  \
  X(EV_CALL_SAME_REV, ZKE_ASSERT, "callop.py:140-151 stay in the caller: reversible_write_counter + 3") \
  X(EV_CALL_SAME_CALL_ID, ZKE_ASSERT, "callop.py:140-151 stay in the caller: call_id same")          \
  X(EV_CALL_SAME_IS_ROOT, ZKE_ASSERT, "callop.py:140-151 stay in the caller: is_root same")          \
  X(EV_CALL_SAME_IS_CREATE, ZKE_ASSERT, "callop.py:140-151 stay in the caller: is_create same")      \
  X(EV_CALL_SAME_CODE_HASH, ZKE_ASSERT, "callop.py:140-151 stay in the caller: code_hash same")      \
  X(EV_CALL_PRECOMPILE, ZKE_NOTIMPL, "callop.py:158-277 call to a precompile: needs StepState.aux_data, which this build's 13-cell step layout does not carry (DESIGN.md)") \
  X(EV_CALL_SAVE0_UNSAT, ZKE_UNSAT, "callop.py:280-297 call_context_lookup(ProgramCounter, Write) unsat") \
  X(EV_CALL_SAVE0_AMBIG, ZKE_AMBIG, "callop.py:280-297 call_context_lookup(ProgramCounter, Write) ambiguous") \
  X(EV_CALL_SAVE0_TYPE, ZKE_ASSERT, "callop.py:280-297 call_context_lookup(ProgramCounter, Write): .value() of a Word") \
  X(EV_CALL_SAVE0_EQ, ZKE_ASSERT, "callop.py:294-297 saved ProgramCounter")                          \
  X(EV_CALL_SAVE1_UNSAT, ZKE_UNSAT, "callop.py:280-297 call_context_lookup(StackPointer, Write) unsat") \
  X(EV_CALL_SAVE1_AMBIG, ZKE_AMBIG, "callop.py:280-297 call_context_lookup(StackPointer, Write) ambiguous") \
  X(EV_CALL_SAVE1_TYPE, ZKE_ASSERT, "callop.py:280-297 call_context_lookup(StackPointer, Write): .value() of a Word") \
  X(EV_CALL_SAVE1_EQ, ZKE_ASSERT, "callop.py:294-297 saved StackPointer")                            \
  X(EV_CALL_SAVE2_UNSAT, ZKE_UNSAT, "callop.py:280-297 call_context_lookup(GasLeft, Write) unsat")   \
  X(EV_CALL_SAVE2_AMBIG, ZKE_AMBIG, "callop.py:280-297 call_context_lookup(GasLeft, Write) ambiguous") \
  X(EV_CALL_SAVE2_TYPE, ZKE_ASSERT, "callop.py:280-297 call_context_lookup(GasLeft, Write): .value() of a Word") \
  X(EV_CALL_SAVE2_EQ, ZKE_ASSERT, "callop.py:294-297 saved GasLeft")                                 \
  X(EV_CALL_SAVE3_UNSAT, ZKE_UNSAT, "callop.py:280-297 call_context_lookup(MemorySize, Write) unsat") \
  X(EV_CALL_SAVE3_AMBIG, ZKE_AMBIG, "callop.py:280-297 call_context_lookup(MemorySize, Write) ambiguous") \
  X(EV_CALL_SAVE3_TYPE, ZKE_ASSERT, "callop.py:280-297 call_context_lookup(MemorySize, Write): .value() of a Word") \
  X(EV_CALL_SAVE3_EQ, ZKE_ASSERT, "callop.py:294-297 saved MemorySize")                              \
  X(EV_CALL_SAVE4_UNSAT, ZKE_UNSAT, "callop.py:280-297 call_context_lookup(ReversibleWriteCounter, Write) unsat") \
  X(EV_CALL_SAVE4_AMBIG, ZKE_AMBIG, "callop.py:280-297 call_context_lookup(ReversibleWriteCounter, Write) ambiguous") \
  X(EV_CALL_SAVE4_TYPE, ZKE_ASSERT, "callop.py:280-297 call_context_lookup(ReversibleWriteCounter, Write): .value() of a Word") \
  X(EV_CALL_SAVE4_EQ, ZKE_ASSERT, "callop.py:294-297 saved ReversibleWriteCounter")                  \
  X(EV_CALL_CTX0_UNSAT, ZKE_UNSAT, "callop.py:301-330 call_context_lookup_word(CallerId, callee) unsat") \
  X(EV_CALL_CTX0_AMBIG, ZKE_AMBIG, "callop.py:301-330 call_context_lookup_word(CallerId, callee) ambiguous") \
  X(EV_CALL_CTX0_EQ, ZKE_ASSERT, "callop.py:327-330 callee CallerId")                                \
  X(EV_CALL_CTX1_UNSAT, ZKE_UNSAT, "callop.py:301-330 call_context_lookup_word(TxId, callee) unsat") \
  X(EV_CALL_CTX1_AMBIG, ZKE_AMBIG, "callop.py:301-330 call_context_lookup_word(TxId, callee) ambiguous") \
  X(EV_CALL_CTX1_EQ, ZKE_ASSERT, "callop.py:327-330 callee TxId")                                    \
  X(EV_CALL_CTX2_UNSAT, ZKE_UNSAT, "callop.py:301-330 call_context_lookup_word(Depth, callee) unsat") \
  X(EV_CALL_CTX2_AMBIG, ZKE_AMBIG, "callop.py:301-330 call_context_lookup_word(Depth, callee) ambiguous") \
  X(EV_CALL_CTX2_EQ, ZKE_ASSERT, "callop.py:327-330 callee Depth")                                   \
  X(EV_CALL_CTX3_UNSAT, ZKE_UNSAT, "callop.py:301-330 call_context_lookup_word(CallerAddress, callee) unsat") \
  X(EV_CALL_CTX3_AMBIG, ZKE_AMBIG, "callop.py:301-330 call_context_lookup_word(CallerAddress, callee) ambiguous") \
  X(EV_CALL_CTX3_EQ, ZKE_ASSERT, "callop.py:327-330 callee CallerAddress")                           \
  X(EV_CALL_CTX4_UNSAT, ZKE_UNSAT, "callop.py:301-330 call_context_lookup_word(CalleeAddress, callee) unsat") \
  X(EV_CALL_CTX4_AMBIG, ZKE_AMBIG, "callop.py:301-330 call_context_lookup_word(CalleeAddress, callee) ambiguous") \
  X(EV_CALL_CTX4_EQ, ZKE_ASSERT, "callop.py:327-330 callee CalleeAddress")                           \
  X(EV_CALL_CTX5_UNSAT, ZKE_UNSAT, "callop.py:301-330 call_context_lookup_word(CallDataOffset, callee) unsat") \
  X(EV_CALL_CTX5_AMBIG, ZKE_AMBIG, "callop.py:301-330 call_context_lookup_word(CallDataOffset, callee) ambiguous") \
  X(EV_CALL_CTX5_EQ, ZKE_ASSERT, "callop.py:327-330 callee CallDataOffset")                          \
  X(EV_CALL_CTX6_UNSAT, ZKE_UNSAT, "callop.py:301-330 call_context_lookup_word(CallDataLength, callee) unsat") \
  X(EV_CALL_CTX6_AMBIG, ZKE_AMBIG, "callop.py:301-330 call_context_lookup_word(CallDataLength, callee) ambiguous") \
  X(EV_CALL_CTX6_EQ, ZKE_ASSERT, "callop.py:327-330 callee CallDataLength")                          \
  X(EV_CALL_CTX7_UNSAT, ZKE_UNSAT, "callop.py:301-330 call_context_lookup_word(ReturnDataOffset, callee) unsat") \
  X(EV_CALL_CTX7_AMBIG, ZKE_AMBIG, "callop.py:301-330 call_context_lookup_word(ReturnDataOffset, callee) ambiguous") \
  X(EV_CALL_CTX7_EQ, ZKE_ASSERT, "callop.py:327-330 callee ReturnDataOffset")                        \
  X(EV_CALL_CTX8_UNSAT, ZKE_UNSAT, "callop.py:301-330 call_context_lookup_word(ReturnDataLength, callee) unsat") \
  X(EV_CALL_CTX8_AMBIG, ZKE_AMBIG, "callop.py:301-330 call_context_lookup_word(ReturnDataLength, callee) ambiguous") \
  X(EV_CALL_CTX8_EQ, ZKE_ASSERT, "callop.py:327-330 callee ReturnDataLength")                        \
  X(EV_CALL_CTX9_UNSAT, ZKE_UNSAT, "callop.py:301-330 call_context_lookup_word(Value, callee) unsat") \
  X(EV_CALL_CTX9_AMBIG, ZKE_AMBIG, "callop.py:301-330 call_context_lookup_word(Value, callee) ambiguous") \
  X(EV_CALL_CTX9_EQ, ZKE_ASSERT, "callop.py:327-330 callee Value")                                   \
  X(EV_CALL_CTX10_UNSAT, ZKE_UNSAT, "callop.py:301-330 call_context_lookup_word(IsSuccess, callee) unsat") \
  X(EV_CALL_CTX10_AMBIG, ZKE_AMBIG, "callop.py:301-330 call_context_lookup_word(IsSuccess, callee) ambiguous") \
  X(EV_CALL_CTX10_EQ, ZKE_ASSERT, "callop.py:327-330 callee IsSuccess")                              \
  X(EV_CALL_CTX11_UNSAT, ZKE_UNSAT, "callop.py:301-330 call_context_lookup_word(IsStatic, callee) unsat") \
  X(EV_CALL_CTX11_AMBIG, ZKE_AMBIG, "callop.py:301-330 call_context_lookup_word(IsStatic, callee) ambiguous") \
  X(EV_CALL_CTX11_EQ, ZKE_ASSERT, "callop.py:327-330 callee IsStatic")                               \
  X(EV_CALL_CTX12_UNSAT, ZKE_UNSAT, "callop.py:301-330 call_context_lookup_word(LastCalleeId, callee) unsat") \
  X(EV_CALL_CTX12_AMBIG, ZKE_AMBIG, "callop.py:301-330 call_context_lookup_word(LastCalleeId, callee) ambiguous") \
  X(EV_CALL_CTX12_EQ, ZKE_ASSERT, "callop.py:327-330 callee LastCalleeId")                           \
  X(EV_CALL_CTX13_UNSAT, ZKE_UNSAT, "callop.py:301-330 call_context_lookup_word(LastCalleeReturnDataOffset, callee) unsat") \
  X(EV_CALL_CTX13_AMBIG, ZKE_AMBIG, "callop.py:301-330 call_context_lookup_word(LastCalleeReturnDataOffset, callee) ambiguous") \
  X(EV_CALL_CTX13_EQ, ZKE_ASSERT, "callop.py:327-330 callee LastCalleeReturnDataOffset")             \
  X(EV_CALL_CTX14_UNSAT, ZKE_UNSAT, "callop.py:301-330 call_context_lookup_word(LastCalleeReturnDataLength, callee) unsat") \
  X(EV_CALL_CTX14_AMBIG, ZKE_AMBIG, "callop.py:301-330 call_context_lookup_word(LastCalleeReturnDataLength, callee) ambiguous") \
  X(EV_CALL_CTX14_EQ, ZKE_ASSERT, "callop.py:327-330 callee LastCalleeReturnDataLength")             \
  X(EV_CALL_CTX15_UNSAT, ZKE_UNSAT, "callop.py:301-330 call_context_lookup_word(IsRoot, callee) unsat") \
  X(EV_CALL_CTX15_AMBIG, ZKE_AMBIG, "callop.py:301-330 call_context_lookup_word(IsRoot, callee) ambiguous") \
  X(EV_CALL_CTX15_EQ, ZKE_ASSERT, "callop.py:327-330 callee IsRoot")                                 \
  X(EV_CALL_CTX16_UNSAT, ZKE_UNSAT, "callop.py:301-330 call_context_lookup_word(IsCreate, callee) unsat") \
  X(EV_CALL_CTX16_AMBIG, ZKE_AMBIG, "callop.py:301-330 call_context_lookup_word(IsCreate, callee) ambiguous") \
  X(EV_CALL_CTX16_EQ, ZKE_ASSERT, "callop.py:327-330 callee IsCreate")                               \
  X(EV_CALL_CTX17_UNSAT, ZKE_UNSAT, "callop.py:301-330 call_context_lookup_word(CodeHash, callee) unsat") \
  X(EV_CALL_CTX17_AMBIG, ZKE_AMBIG, "callop.py:301-330 call_context_lookup_word(CodeHash, callee) ambiguous") \
  X(EV_CALL_CTX17_EQ, ZKE_ASSERT, "callop.py:327-330 callee CodeHash")                               \
  X(EV_CALL_VALUE_WORD, ZKE_ASSERT, "callop.py:313 select_word: a half of the value >= 2^128")       \
  X(EV_CALL_NC_RWC, ZKE_ASSERT, "callop.py:335-344 new context: rw_counter delta")                   \
  X(EV_CALL_NC_CALL_ID, ZKE_ASSERT, "callop.py:335-344 new context: call_id to the callee's")        \
  X(EV_CALL_NC_IS_ROOT, ZKE_ASSERT, "callop.py:335-344 new context: is_root to False")               \
  X(EV_CALL_NC_IS_CREATE, ZKE_ASSERT, "callop.py:335-344 new context: is_create to False")           \
  X(EV_CALL_NC_CODE_HASH, ZKE_ASSERT, "callop.py:335-344 new context: code_hash to the callee's")    \
  X(EV_CALL_NC_GAS, ZKE_ASSERT, "callop.py:335-344 new context: gas_left to the callee's")           \
  X(EV_CALL_NC_REV, ZKE_ASSERT, "callop.py:335-344 new context: reversible_write_counter to 2")      \
  X(EV_CALL_NC_LOG, ZKE_ASSERT, "callop.py:335-344 new context: log_id same")                        \
  X(EV_CALL_NC_PC, ZKE_ASSERT, "callop.py:335-344 new context: program_counter to 0")                \
  X(EV_CALL_NC_SP, ZKE_ASSERT, "callop.py:335-344 new context: stack_pointer to 1024")               \
  X(EV_CALL_NC_MEM, ZKE_ASSERT, "callop.py:335-344 new context: memory_word_size to 0") \
  X(EV_CR_RESP_OPCODE, ZKE_UNSAT, "create.py:24 responsible_opcode_lookup(opcode)") \
  X(EV_CR_POP0_UNSAT, ZKE_UNSAT, "create.py:30-33 stack_pop value unsat") \
  X(EV_CR_POP0_AMBIG, ZKE_AMBIG, "create.py:30-33 stack_pop value ambiguous") \
  X(EV_CR_POP1_UNSAT, ZKE_UNSAT, "create.py:30-33 stack_pop offset unsat") \
  X(EV_CR_POP1_AMBIG, ZKE_AMBIG, "create.py:30-33 stack_pop offset ambiguous") \
  X(EV_CR_POP2_UNSAT, ZKE_UNSAT, "create.py:30-33 stack_pop size unsat") \
  X(EV_CR_POP2_AMBIG, ZKE_AMBIG, "create.py:30-33 stack_pop size ambiguous") \
  X(EV_CR_POP3_UNSAT, ZKE_UNSAT, "create.py:30-33 stack_pop salt (CREATE2) unsat") \
  X(EV_CR_POP3_AMBIG, ZKE_AMBIG, "create.py:30-33 stack_pop salt (CREATE2) ambiguous") \
  X(EV_CR_PUSH_UNSAT, ZKE_UNSAT, "create.py:34 stack_push contract address unsat") \
  X(EV_CR_PUSH_AMBIG, ZKE_AMBIG, "create.py:34 stack_push contract address ambiguous") \
  X(EV_CR_OFF_DOMAIN, ZKE_VALUE, "create.py:36 word_to_fq(offset, 5): word_to_fq of a half >= 2^128 -> OverflowError") \
  X(EV_CR_OFF_RANGE, ZKE_RANGE, "create.py:36 word_to_fq(offset, 5): more than 5 bytes") \
  X(EV_CR_SIZE_DOMAIN, ZKE_VALUE, "create.py:37 word_to_fq(size, 5): word_to_fq of a half >= 2^128 -> OverflowError") \
  X(EV_CR_SIZE_RANGE, ZKE_RANGE, "create.py:37 word_to_fq(size, 5): more than 5 bytes") \
  X(EV_CR_DEPTH_UNSAT, ZKE_UNSAT, "create.py:39 call_context_lookup(Depth) unsat") \
  X(EV_CR_DEPTH_AMBIG, ZKE_AMBIG, "create.py:39 call_context_lookup(Depth) ambiguous") \
  X(EV_CR_DEPTH_TYPE, ZKE_ASSERT, "create.py:39 call_context_lookup(Depth): .value() of a Word") \
  X(EV_CR_TXID_UNSAT, ZKE_UNSAT, "create.py:40 call_context_lookup(TxId) unsat") \
  X(EV_CR_TXID_AMBIG, ZKE_AMBIG, "create.py:40 call_context_lookup(TxId) ambiguous") \
  X(EV_CR_TXID_TYPE, ZKE_ASSERT, "create.py:40 call_context_lookup(TxId): .value() of a Word") \
  X(EV_CR_CALLER_UNSAT, ZKE_UNSAT, "create.py:41 call_context_lookup_word(CallerAddress) unsat") \
  X(EV_CR_CALLER_AMBIG, ZKE_AMBIG, "create.py:41 call_context_lookup_word(CallerAddress) ambiguous") \
  X(EV_CR_CALLER_DOMAIN, ZKE_VALUE, "create.py:42 word_to_address(caller address): word_to_fq of a half >= 2^128 -> OverflowError") \
  X(EV_CR_CALLER_RANGE, ZKE_RANGE, "create.py:42 word_to_address(caller address): more than 20 bytes") \
  X(EV_CR_NONCE_UNSAT, ZKE_UNSAT, "create.py:43 account_write(caller, Nonce) unsat") \
  X(EV_CR_NONCE_AMBIG, ZKE_AMBIG, "create.py:43 account_write(caller, Nonce) ambiguous") \
  X(EV_CR_NONCE_TYPE, ZKE_ASSERT, "create.py:43 account_write(caller, Nonce): .value() of a Word") \
  X(EV_CR_NONCE_PREV_TYPE, ZKE_ASSERT, "create.py:43 account_write(caller, Nonce): value_prev.value() of a Word") \
  X(EV_CR_BAL_UNSAT, ZKE_UNSAT, "create.py:44 account_read(caller, Balance) unsat") \
  X(EV_CR_BAL_AMBIG, ZKE_AMBIG, "create.py:44 account_read(caller, Balance) ambiguous") \
  X(EV_CR_BAL_TYPE, ZKE_ASSERT, "create.py:44 account_read(caller, Balance): .value() of a Word") \
  X(EV_CR_SUCCESS_UNSAT, ZKE_UNSAT, "create.py:45 call_context_lookup(IsSuccess) unsat") \
  X(EV_CR_SUCCESS_AMBIG, ZKE_AMBIG, "create.py:45 call_context_lookup(IsSuccess) ambiguous") \
  X(EV_CR_SUCCESS_TYPE, ZKE_ASSERT, "create.py:45 call_context_lookup(IsSuccess): .value() of a Word") \
  X(EV_CR_STATIC_UNSAT, ZKE_UNSAT, "create.py:46 call_context_lookup(IsStatic) unsat") \
  X(EV_CR_STATIC_AMBIG, ZKE_AMBIG, "create.py:46 call_context_lookup(IsStatic) ambiguous") \
  X(EV_CR_STATIC_TYPE, ZKE_ASSERT, "create.py:46 call_context_lookup(IsStatic): .value() of a Word") \
  X(EV_CR_REVEND_UNSAT, ZKE_UNSAT, "create.py:47 reversion_info: RwCounterEndOfReversion unsat") \
  X(EV_CR_REVEND_AMBIG, ZKE_AMBIG, "create.py:47 reversion_info: RwCounterEndOfReversion ambiguous") \
  X(EV_CR_REVEND_TYPE, ZKE_ASSERT, "create.py:47 reversion_info: RwCounterEndOfReversion: .value() of a Word") \
  X(EV_CR_PERSIST_UNSAT, ZKE_UNSAT, "create.py:47 reversion_info: IsPersistent unsat") \
  X(EV_CR_PERSIST_AMBIG, ZKE_AMBIG, "create.py:47 reversion_info: IsPersistent ambiguous") \
  X(EV_CR_PERSIST_TYPE, ZKE_ASSERT, "create.py:47 reversion_info: IsPersistent: .value() of a Word") \
  X(EV_CR_MEMSIZE_RANGE, ZKE_RANGE, "create.py:59-62 memory_expansion: memory size beyond 4 bytes") \
  X(EV_CR_MEM_MAX, ZKE_ASSERT, "create.py:59-62 memory_expansion: max(): curr.memory_word_size beyond 4 bytes") \
  X(EV_CR_WORDLEN_RANGE, ZKE_RANGE, "create.py:68 constant_divmod(size + 31, 32, 4): quotient beyond 4 bytes") \
  X(EV_CR_GAS_64TH_RANGE, ZKE_RANGE, "create.py:76 constant_divmod(gas_available, 64, 8): quotient beyond 8 bytes") \
  X(EV_CR_GAS_MIN_RANGE, ZKE_ASSERT, "create.py:81-85 min(all_but_one_64th_gas, gas_left, 8): an operand beyond 8 bytes") \
  X(EV_CR_DEPTH_RANGE, ZKE_ASSERT, "create.py:89 compare(depth, 1025, 2): depth beyond 2 bytes") \
  X(EV_CR_BAL_CMP_RANGE, ZKE_ASSERT, "create.py:91 compare_word(balance, value): a half of the value >= 2^128") \
  X(EV_CR_NONCE_RANGE, ZKE_ASSERT, "create.py:93 compare(nonce_prev, MAX_U64, 8): nonce_prev beyond 8 bytes") \
  X(EV_CR_AUX_MISSING, ZKE_ASSERT, "create.py:107 curr.aux_data (the init code's hash): not exactly one entry for this step in the step-aux table") \
  X(EV_CR_ADDR2_DOMAIN, ZKE_VALUE, "instruction.py:1349-1350 salt / code hash .to_bytes(32): a half makes the integer >= 2^256 -> OverflowError") \
  X(EV_CR_AL_UNSAT, ZKE_UNSAT, "create.py:116 add_account_to_access_list(tx_id, contract_address) unsat") \
  X(EV_CR_AL_AMBIG, ZKE_AMBIG, "create.py:116 add_account_to_access_list(tx_id, contract_address) ambiguous") \
  X(EV_CR_AL_PREV_TYPE, ZKE_ASSERT, "instruction.py:1057 value_prev.value() of a Word") \
  X(EV_CR_CHASH_UNSAT, ZKE_UNSAT, "create.py:120 account_read_word(contract, CodeHash) unsat") \
  X(EV_CR_CHASH_AMBIG, ZKE_AMBIG, "create.py:120 account_read_word(contract, CodeHash) ambiguous") \
  X(EV_CR_CNONCE_UNSAT, ZKE_UNSAT, "create.py:121 account_read(contract, Nonce) unsat") \
  X(EV_CR_CNONCE_AMBIG, ZKE_AMBIG, "create.py:121 account_read(contract, Nonce) ambiguous") \
  X(EV_CR_CNONCE_TYPE, ZKE_ASSERT, "create.py:121 account_read(contract, Nonce): .value() of a Word") \
  X(EV_CR_RETURN_DOMAIN, ZKE_VALUE, "create.py:130 word_to_fq(return address word, 20): word_to_fq of a half >= 2^128 -> OverflowError") \
  X(EV_CR_RETURN_RANGE, ZKE_RANGE, "create.py:130 word_to_fq(return address word, 20): more than 20 bytes") \
  X(EV_CR_RETURN_EQ, ZKE_ASSERT, "create.py:129-132 pushed address == is_success * contract_address") \
  X(EV_CR_CREVEND_UNSAT, ZKE_UNSAT, "create.py:135 reversion_info(callee): RwCounterEndOfReversion unsat") \
  X(EV_CR_CREVEND_AMBIG, ZKE_AMBIG, "create.py:135 reversion_info(callee): RwCounterEndOfReversion ambiguous") \
  X(EV_CR_CREVEND_TYPE, ZKE_ASSERT, "create.py:135 reversion_info(callee): RwCounterEndOfReversion: .value() of a Word") \
  X(EV_CR_CPERSIST_UNSAT, ZKE_UNSAT, "create.py:135 reversion_info(callee): IsPersistent unsat") \
  X(EV_CR_CPERSIST_AMBIG, ZKE_AMBIG, "create.py:135 reversion_info(callee): IsPersistent ambiguous") \
  X(EV_CR_CPERSIST_TYPE, ZKE_ASSERT, "create.py:135 reversion_info(callee): IsPersistent: .value() of a Word") \
  X(EV_CR_CPERSIST_EQ, ZKE_ASSERT, "create.py:136-139 callee is_persistent == is_persistent * is_success") \
  X(EV_CR_SEND_UNSAT, ZKE_UNSAT, "create.py:142-144 transfer: sub_balance(caller) unsat") \
  X(EV_CR_SEND_AMBIG, ZKE_AMBIG, "create.py:142-144 transfer: sub_balance(caller) ambiguous") \
  X(EV_CR_SEND_REV_UNSAT, ZKE_UNSAT, "create.py:142-144 transfer: sub_balance(caller): reversion row unsat") \
  X(EV_CR_SEND_REV_AMBIG, ZKE_AMBIG, "create.py:142-144 transfer: sub_balance(caller): reversion row ambiguous") \
  X(EV_CR_SEND_EQ, ZKE_ASSERT, "create.py:142-144 transfer: sub_balance(caller): balance_prev / balance == add_words(..)") \
  X(EV_CR_SEND_CARRY, ZKE_ASSERT, "create.py:142-144 transfer: sub_balance(caller): carry == 0") \
  X(EV_CR_RECV_UNSAT, ZKE_UNSAT, "create.py:142-144 transfer: add_balance(contract) unsat") \
  X(EV_CR_RECV_AMBIG, ZKE_AMBIG, "create.py:142-144 transfer: add_balance(contract) ambiguous") \
  X(EV_CR_RECV_REV_UNSAT, ZKE_UNSAT, "create.py:142-144 transfer: add_balance(contract): reversion row unsat") \
  X(EV_CR_RECV_REV_AMBIG, ZKE_AMBIG, "create.py:142-144 transfer: add_balance(contract): reversion row ambiguous") \
  X(EV_CR_RECV_EQ, ZKE_ASSERT, "create.py:142-144 transfer: add_balance(contract): balance_prev / balance == add_words(..)") \
  X(EV_CR_RECV_CARRY, ZKE_ASSERT, "create.py:142-144 transfer: add_balance(contract): carry == 0") \
  X(EV_CR_NEWNONCE_UNSAT, ZKE_UNSAT, "create.py:147 account_write(contract, Nonce) unsat") \
  X(EV_CR_NEWNONCE_AMBIG, ZKE_AMBIG, "create.py:147 account_write(contract, Nonce) ambiguous") \
  X(EV_CR_NEWNONCE_TYPE, ZKE_ASSERT, "create.py:147 account_write(contract, Nonce): .value() of a Word") \
  X(EV_CR_NEWNONCE_PREV_TYPE, ZKE_ASSERT, "create.py:147 account_write(contract, Nonce): value_prev.value() of a Word") \
  X(EV_CR_NEWNONCE_EQ, ZKE_ASSERT, "create.py:148 EIP-161: the new contract's nonce == 1") \
  X(EV_CR_COPY_UNSAT, ZKE_UNSAT, "create.py:152-162 copy_lookup(memory -> bytecode next.code_hash) unsat") \
  X(EV_CR_COPY_AMBIG, ZKE_AMBIG, "create.py:152-162 copy_lookup(memory -> bytecode next.code_hash) ambiguous") \
  X(EV_CR_CODE_LEN_UNSAT, ZKE_UNSAT, "create.py:166 bytecode_length(next.code_hash) unsat") \
  X(EV_CR_CODE_LEN_AMBIG, ZKE_AMBIG, "create.py:166 bytecode_length(next.code_hash) ambiguous") \
  X(EV_CR_CODE_LEN_EQ, ZKE_ASSERT, "create.py:167 code_size == size") \
  X(EV_CR_SAVE0_UNSAT, ZKE_UNSAT, "create.py:170-186 call_context_lookup(ProgramCounter, Write) unsat") \
  X(EV_CR_SAVE0_AMBIG, ZKE_AMBIG, "create.py:170-186 call_context_lookup(ProgramCounter, Write) ambiguous") \
  X(EV_CR_SAVE0_TYPE, ZKE_ASSERT, "create.py:170-186 call_context_lookup(ProgramCounter, Write): .value() of a Word") \
  X(EV_CR_SAVE0_EQ, ZKE_ASSERT, "create.py:183-186 saved ProgramCounter") \
  X(EV_CR_SAVE1_UNSAT, ZKE_UNSAT, "create.py:170-186 call_context_lookup(StackPointer, Write) unsat") \
  X(EV_CR_SAVE1_AMBIG, ZKE_AMBIG, "create.py:170-186 call_context_lookup(StackPointer, Write) ambiguous") \
  X(EV_CR_SAVE1_TYPE, ZKE_ASSERT, "create.py:170-186 call_context_lookup(StackPointer, Write): .value() of a Word") \
  X(EV_CR_SAVE1_EQ, ZKE_ASSERT, "create.py:183-186 saved StackPointer") \
  X(EV_CR_SAVE2_UNSAT, ZKE_UNSAT, "create.py:170-186 call_context_lookup(GasLeft, Write) unsat") \
  X(EV_CR_SAVE2_AMBIG, ZKE_AMBIG, "create.py:170-186 call_context_lookup(GasLeft, Write) ambiguous") \
  X(EV_CR_SAVE2_TYPE, ZKE_ASSERT, "create.py:170-186 call_context_lookup(GasLeft, Write): .value() of a Word") \
  X(EV_CR_SAVE2_EQ, ZKE_ASSERT, "create.py:183-186 saved GasLeft") \
  X(EV_CR_SAVE3_UNSAT, ZKE_UNSAT, "create.py:170-186 call_context_lookup(MemorySize, Write) unsat") \
  X(EV_CR_SAVE3_AMBIG, ZKE_AMBIG, "create.py:170-186 call_context_lookup(MemorySize, Write) ambiguous") \
  X(EV_CR_SAVE3_TYPE, ZKE_ASSERT, "create.py:170-186 call_context_lookup(MemorySize, Write): .value() of a Word") \
  X(EV_CR_SAVE3_EQ, ZKE_ASSERT, "create.py:183-186 saved MemorySize") \
  X(EV_CR_SAVE4_UNSAT, ZKE_UNSAT, "create.py:170-186 call_context_lookup(ReversibleWriteCounter, Write) unsat") \
  X(EV_CR_SAVE4_AMBIG, ZKE_AMBIG, "create.py:170-186 call_context_lookup(ReversibleWriteCounter, Write) ambiguous") \
  X(EV_CR_SAVE4_TYPE, ZKE_ASSERT, "create.py:170-186 call_context_lookup(ReversibleWriteCounter, Write): .value() of a Word") \
  X(EV_CR_SAVE4_EQ, ZKE_ASSERT, "create.py:183-186 saved ReversibleWriteCounter") \
  X(EV_CR_CTX0_UNSAT, ZKE_UNSAT, "create.py:188-211 call_context_lookup_word(CallerId, callee) unsat") \
  X(EV_CR_CTX0_AMBIG, ZKE_AMBIG, "create.py:188-211 call_context_lookup_word(CallerId, callee) ambiguous") \
  X(EV_CR_CTX0_EQ, ZKE_ASSERT, "create.py:202-211 callee CallerId") \
  X(EV_CR_CTX1_UNSAT, ZKE_UNSAT, "create.py:188-211 call_context_lookup_word(TxId, callee) unsat") \
  X(EV_CR_CTX1_AMBIG, ZKE_AMBIG, "create.py:188-211 call_context_lookup_word(TxId, callee) ambiguous") \
  X(EV_CR_CTX1_EQ, ZKE_ASSERT, "create.py:202-211 callee TxId") \
  X(EV_CR_CTX2_UNSAT, ZKE_UNSAT, "create.py:188-211 call_context_lookup_word(Depth, callee) unsat") \
  X(EV_CR_CTX2_AMBIG, ZKE_AMBIG, "create.py:188-211 call_context_lookup_word(Depth, callee) ambiguous") \
  X(EV_CR_CTX2_EQ, ZKE_ASSERT, "create.py:202-211 callee Depth") \
  X(EV_CR_CTX3_UNSAT, ZKE_UNSAT, "create.py:188-211 call_context_lookup_word(CallerAddress, callee) unsat") \
  X(EV_CR_CTX3_AMBIG, ZKE_AMBIG, "create.py:188-211 call_context_lookup_word(CallerAddress, callee) ambiguous") \
  X(EV_CR_CTX3_EQ, ZKE_ASSERT, "create.py:202-211 callee CallerAddress") \
  X(EV_CR_CTX4_UNSAT, ZKE_UNSAT, "create.py:188-211 call_context_lookup_word(CalleeAddress, callee) unsat") \
  X(EV_CR_CTX4_AMBIG, ZKE_AMBIG, "create.py:188-211 call_context_lookup_word(CalleeAddress, callee) ambiguous") \
  X(EV_CR_CTX4_EQ, ZKE_ASSERT, "create.py:202-211 callee CalleeAddress") \
  X(EV_CR_CTX5_UNSAT, ZKE_UNSAT, "create.py:188-211 call_context_lookup_word(IsSuccess, callee) unsat") \
  X(EV_CR_CTX5_AMBIG, ZKE_AMBIG, "create.py:188-211 call_context_lookup_word(IsSuccess, callee) ambiguous") \
  X(EV_CR_CTX5_EQ, ZKE_ASSERT, "create.py:202-211 callee IsSuccess") \
  X(EV_CR_CTX6_UNSAT, ZKE_UNSAT, "create.py:188-211 call_context_lookup_word(IsStatic, callee) unsat") \
  X(EV_CR_CTX6_AMBIG, ZKE_AMBIG, "create.py:188-211 call_context_lookup_word(IsStatic, callee) ambiguous") \
  X(EV_CR_CTX6_EQ, ZKE_ASSERT, "create.py:202-211 callee IsStatic") \
  X(EV_CR_CTX7_UNSAT, ZKE_UNSAT, "create.py:188-211 call_context_lookup_word(IsRoot, callee) unsat") \
  X(EV_CR_CTX7_AMBIG, ZKE_AMBIG, "create.py:188-211 call_context_lookup_word(IsRoot, callee) ambiguous") \
  X(EV_CR_CTX7_EQ, ZKE_ASSERT, "create.py:202-211 callee IsRoot") \
  X(EV_CR_CTX8_UNSAT, ZKE_UNSAT, "create.py:188-211 call_context_lookup_word(IsCreate, callee) unsat") \
  X(EV_CR_CTX8_AMBIG, ZKE_AMBIG, "create.py:188-211 call_context_lookup_word(IsCreate, callee) ambiguous") \
  X(EV_CR_CTX8_EQ, ZKE_ASSERT, "create.py:202-211 callee IsCreate") \
  X(EV_CR_CTX9_UNSAT, ZKE_UNSAT, "create.py:188-211 call_context_lookup_word(CodeHash, callee) unsat") \
  X(EV_CR_CTX9_AMBIG, ZKE_AMBIG, "create.py:188-211 call_context_lookup_word(CodeHash, callee) ambiguous") \
  X(EV_CR_CTX9_EQ, ZKE_ASSERT, "create.py:202-211 callee CodeHash") \
  X(EV_CR_NC_RWC, ZKE_ASSERT, "create.py:213-223 new context: rw_counter delta") \
  X(EV_CR_NC_CALL_ID, ZKE_ASSERT, "create.py:213-223 new context: call_id to the callee's") \
  X(EV_CR_NC_IS_ROOT, ZKE_ASSERT, "create.py:213-223 new context: is_root to False") \
  X(EV_CR_NC_IS_CREATE, ZKE_ASSERT, "create.py:213-223 new context: is_create to True") \
  X(EV_CR_NC_GAS, ZKE_ASSERT, "create.py:213-223 new context: gas_left to the callee's") \
  X(EV_CR_NC_REV, ZKE_ASSERT, "create.py:213-223 new context: reversible_write_counter to 3") \
  X(EV_CR_NC_LOG, ZKE_ASSERT, "create.py:213-223 new context: log_id same") \
  X(EV_CR_NC_PC, ZKE_ASSERT, "create.py:213-223 new context: program_counter to 0") \
  X(EV_CR_NC_SP, ZKE_ASSERT, "create.py:213-223 new context: stack_pointer to 1024") \
  X(EV_CR_NC_MEM, ZKE_ASSERT, "create.py:213-223 new context: memory_word_size to 0") \
  X(EV_CR_FAIL_SUCCESS, ZKE_ASSERT, "create.py:228 pre-check failure / address collision: is_success == 0") \
  X(EV_CR_LAST0_UNSAT, ZKE_UNSAT, "create.py:230-238 call_context_lookup(LastCalleeId, Write) unsat") \
  X(EV_CR_LAST0_AMBIG, ZKE_AMBIG, "create.py:230-238 call_context_lookup(LastCalleeId, Write) ambiguous") \
  X(EV_CR_LAST0_TYPE, ZKE_ASSERT, "create.py:230-238 call_context_lookup(LastCalleeId, Write): .value() of a Word") \
  X(EV_CR_LAST0_EQ, ZKE_ASSERT, "create.py:235-238 LastCalleeId == 0") \
  X(EV_CR_LAST1_UNSAT, ZKE_UNSAT, "create.py:230-238 call_context_lookup(LastCalleeReturnDataOffset, Write) unsat") \
  X(EV_CR_LAST1_AMBIG, ZKE_AMBIG, "create.py:230-238 call_context_lookup(LastCalleeReturnDataOffset, Write) ambiguous") \
  X(EV_CR_LAST1_TYPE, ZKE_ASSERT, "create.py:230-238 call_context_lookup(LastCalleeReturnDataOffset, Write): .value() of a Word") \
  X(EV_CR_LAST1_EQ, ZKE_ASSERT, "create.py:235-238 LastCalleeReturnDataOffset == 0") \
  X(EV_CR_LAST2_UNSAT, ZKE_UNSAT, "create.py:230-238 call_context_lookup(LastCalleeReturnDataLength, Write) unsat") \
  X(EV_CR_LAST2_AMBIG, ZKE_AMBIG, "create.py:230-238 call_context_lookup(LastCalleeReturnDataLength, Write) ambiguous") \
  X(EV_CR_LAST2_TYPE, ZKE_ASSERT, "create.py:230-238 call_context_lookup(LastCalleeReturnDataLength, Write): .value() of a Word") \
  X(EV_CR_LAST2_EQ, ZKE_ASSERT, "create.py:235-238 LastCalleeReturnDataLength == 0") \
  X(EV_CR_SAME_RWC, ZKE_ASSERT, "create.py:242-254 same context: rw_counter delta") \
  X(EV_CR_SAME_PC, ZKE_ASSERT, "create.py:242-254 same context: program_counter + 1") \
  X(EV_CR_SAME_SP, ZKE_ASSERT, "create.py:242-254 same context: stack_pointer + 2 (+ 1 for CREATE2)") \
  X(EV_CR_SAME_REV, ZKE_ASSERT, "create.py:242-254 same context: reversible_write_counter + 3 iff created without init code") \
  X(EV_CR_SAME_GAS, ZKE_ASSERT, "create.py:242-254 same context: gas_left - gas_cost") \
  X(EV_CR_SAME_MEM, ZKE_ASSERT, "create.py:242-254 same context: memory_word_size to next_memory_size") \
  X(EV_CR_SAME_CALL_ID, ZKE_ASSERT, "create.py:242-254 same context: call_id same") \
  X(EV_CR_SAME_IS_ROOT, ZKE_ASSERT, "create.py:242-254 same context: is_root same") \
  X(EV_CR_SAME_IS_CREATE, ZKE_ASSERT, "create.py:242-254 same context: is_create same") \
  X(EV_CR_SAME_CODE_HASH, ZKE_ASSERT, "create.py:242-254 same context: code_hash same") \
  X(EV_ESS_OPCODE, ZKE_ASSERT, "error_oog_sload_sstore.py:18-19 is_sstore + is_sload == 1") \
  X(EV_ESS_KEY_UNSAT, ZKE_UNSAT, "error_oog_sload_sstore.py:21 stack_pop storage key unsat") \
  X(EV_ESS_KEY_AMBIG, ZKE_AMBIG, "error_oog_sload_sstore.py:21 stack_pop storage key ambiguous") \
  X(EV_ESS_TXID_UNSAT, ZKE_UNSAT, "error_oog_sload_sstore.py:23 call_context_lookup(TxId) unsat") \
  X(EV_ESS_TXID_AMBIG, ZKE_AMBIG, "error_oog_sload_sstore.py:23 call_context_lookup(TxId) ambiguous") \
  X(EV_ESS_TXID_TYPE, ZKE_ASSERT, "error_oog_sload_sstore.py:23 call_context_lookup(TxId): .value() of a Word") \
  X(EV_ESS_CALLEE_UNSAT, ZKE_UNSAT, "error_oog_sload_sstore.py:24 call_context_lookup_word(CalleeAddress) unsat") \
  X(EV_ESS_CALLEE_AMBIG, ZKE_AMBIG, "error_oog_sload_sstore.py:24 call_context_lookup_word(CalleeAddress) ambiguous") \
  X(EV_ESS_CALLEE_DOMAIN, ZKE_VALUE, "error_oog_sload_sstore.py:25 word_to_address: word_to_fq of a half >= 2^128 -> OverflowError") \
  X(EV_ESS_CALLEE_RANGE, ZKE_RANGE, "error_oog_sload_sstore.py:25 word_to_address: more than 20 bytes") \
  X(EV_ESS_AL_UNSAT, ZKE_UNSAT, "error_oog_sload_sstore.py:26 read_account_storage_to_access_list unsat") \
  X(EV_ESS_AL_AMBIG, ZKE_AMBIG, "error_oog_sload_sstore.py:26 read_account_storage_to_access_list ambiguous") \
  X(EV_ESS_AL_TYPE, ZKE_ASSERT, "error_oog_sload_sstore.py:26 read_account_storage_to_access_list: .value() of a Word") \
  X(EV_ESS_VAL_UNSAT, ZKE_UNSAT, "error_oog_sload_sstore.py:31 stack_pop value (SSTORE) unsat") \
  X(EV_ESS_VAL_AMBIG, ZKE_AMBIG, "error_oog_sload_sstore.py:31 stack_pop value (SSTORE) ambiguous") \
  X(EV_ESS_READ_UNSAT, ZKE_UNSAT, "error_oog_sload_sstore.py:32 account_storage_read (SSTORE) unsat") \
  X(EV_ESS_READ_AMBIG, ZKE_AMBIG, "error_oog_sload_sstore.py:32 account_storage_read (SSTORE) ambiguous") \
  X(EV_ESS_AUX_MISSING, ZKE_ASSERT, "error_oog_sload_sstore.py:33 Word(curr.aux_data): not exactly one entry for this step in the step-aux table") \
  X(EV_ESS_AUX_RANGE, ZKE_ASSERT, "error_oog_sload_sstore.py:33 Word(curr.aux_data): the integer does not fit 32 bytes") \
  X(EV_ESS_GAS_RANGE, ZKE_ASSERT, "error_oog_sload_sstore.py:48 compare(gas_left, gas_cost, 8): gas_left beyond 8 bytes") \
  X(EV_ESS_SLOAD_NOT_OOG, ZKE_ASSERT, "error_oog_sload_sstore.py:50 SLOAD: gas_left < gas_cost") \
  X(EV_ESS_SSTORE_NOT_OOG, ZKE_ASSERT, "error_oog_sload_sstore.py:53-56 SSTORE: gas_left <= 2300 or gas_left < gas_cost") \
  X(EV_EOCR_OPCODE, ZKE_ASSERT, "error_oog_create.py:25 is_create + is_create2 == 1") \
  X(EV_EOCR_OFF_UNSAT, ZKE_UNSAT, "error_oog_create.py:28 stack_lookup(Read, 1) offset unsat") \
  X(EV_EOCR_OFF_AMBIG, ZKE_AMBIG, "error_oog_create.py:28 stack_lookup(Read, 1) offset ambiguous") \
  X(EV_EOCR_SIZE_UNSAT, ZKE_UNSAT, "error_oog_create.py:29 stack_lookup(Read, 2) size unsat") \
  X(EV_EOCR_SIZE_AMBIG, ZKE_AMBIG, "error_oog_create.py:29 stack_lookup(Read, 2) size ambiguous") \
  X(EV_EOCR_SIZE_DOMAIN, ZKE_VALUE, "error_oog_create.py:30 memory_offset_and_length: size: word_to_fq of a half >= 2^128 -> OverflowError") \
  X(EV_EOCR_SIZE_RANGE, ZKE_RANGE, "error_oog_create.py:30 memory_offset_and_length: size: more than 5 bytes") \
  X(EV_EOCR_OFF_DOMAIN, ZKE_VALUE, "error_oog_create.py:30 memory_offset_and_length: offset: word_to_fq of a half >= 2^128 -> OverflowError") \
  X(EV_EOCR_OFF_RANGE, ZKE_RANGE, "error_oog_create.py:30 memory_offset_and_length: offset: more than 5 bytes") \
  X(EV_EOCR_ROOT_UNSAT, ZKE_UNSAT, "error_oog_create.py:32 call_context_lookup(IsRoot) unsat") \
  X(EV_EOCR_ROOT_AMBIG, ZKE_AMBIG, "error_oog_create.py:32 call_context_lookup(IsRoot) ambiguous") \
  X(EV_EOCR_ROOT_TYPE, ZKE_ASSERT, "error_oog_create.py:32 call_context_lookup(IsRoot): .value() of a Word") \
  X(EV_EOCR_TXID_UNSAT, ZKE_UNSAT, "error_oog_create.py:36 call_context_lookup(TxId) unsat") \
  X(EV_EOCR_TXID_AMBIG, ZKE_AMBIG, "error_oog_create.py:36 call_context_lookup(TxId) ambiguous") \
  X(EV_EOCR_TXID_TYPE, ZKE_ASSERT, "error_oog_create.py:36 call_context_lookup(TxId): .value() of a Word") \
  X(EV_EOCR_BYTE_UNSAT, ZKE_UNSAT, "error_oog_create.py:37 tx_calldata_lookup(tx_id, idx) unsat") \
  X(EV_EOCR_BYTE_AMBIG, ZKE_AMBIG, "error_oog_create.py:37 tx_calldata_lookup(tx_id, idx) ambiguous") \
  X(EV_EOCR_BYTE_TYPE, ZKE_ASSERT, "error_oog_create.py:37 tx_calldata_lookup(tx_id, idx): .value() of a Word") \
  X(EV_EOCR_MEMSIZE_RANGE, ZKE_RANGE, "error_oog_create.py:47 memory_expansion: memory size beyond 4 bytes") \
  X(EV_EOCR_MEM_MAX, ZKE_ASSERT, "error_oog_create.py:47 memory_expansion: max(): curr.memory_word_size beyond 4 bytes") \
  X(EV_EOCR_WORDSIZE_RANGE, ZKE_RANGE, "error_oog_create.py:51 constant_divmod(size + 31, 32, 4): quotient beyond 4 bytes") \
  X(EV_EOCR_GAS_RANGE, ZKE_ASSERT, "error_oog_create.py:60 compare(gas_left, gas_cost, 8): gas_left beyond 8 bytes") \
  X(EV_EOCR_NOT_OOG, ZKE_ASSERT, "error_oog_create.py:62 insufficient_gas + is_exceed_max_initcode_size != 0") \
  X(EV_EOPC_CALLEE_UNSAT, ZKE_UNSAT, "error_oog_precompile.py:10 call_context_lookup_word(CalleeAddress) unsat") \
  X(EV_EOPC_CALLEE_AMBIG, ZKE_AMBIG, "error_oog_precompile.py:10 call_context_lookup_word(CalleeAddress) ambiguous") \
  X(EV_EOPC_CALLEE_DOMAIN, ZKE_VALUE, "error_oog_precompile.py:11 word_to_address: word_to_fq of a half >= 2^128 -> OverflowError") \
  X(EV_EOPC_CALLEE_RANGE, ZKE_RANGE, "error_oog_precompile.py:11 word_to_address: more than 20 bytes") \
  X(EV_EOPC_CDLEN_UNSAT, ZKE_UNSAT, "error_oog_precompile.py:12 call_context_lookup(CallDataLength) unsat") \
  X(EV_EOPC_CDLEN_AMBIG, ZKE_AMBIG, "error_oog_precompile.py:12 call_context_lookup(CallDataLength) ambiguous") \
  X(EV_EOPC_CDLEN_TYPE, ZKE_ASSERT, "error_oog_precompile.py:12 call_context_lookup(CallDataLength): .value() of a Word") \
  X(EV_EOPC_NOT_PRECOMPILE, ZKE_ASSERT, "error_oog_precompile.py:15 the callee address is one of the nine precompiles") \
  X(EV_EOPC_WORDSIZE_RANGE, ZKE_RANGE, "error_oog_precompile.py:27 memory_copier_gas_cost: constant_divmod(len + 31, 32, 4): quotient beyond 4 bytes") \
  X(EV_EOPC_GAS_LEFT_RANGE, ZKE_ASSERT, "error_oog_precompile.py:30 compare(gas_left, gas_cost, 8): gas_left beyond 8 bytes") \
  X(EV_EOPC_GAS_INT, ZKE_VALUE, "error_oog_precompile.py:19-30 every precompile but DATACOPY / BN254PAIRING: gas_cost is a Python int, compare() raises AttributeError on it") \
  X(EV_EOPC_GAS_COST_RANGE, ZKE_ASSERT, "error_oog_precompile.py:23-24,30 compare(): gas_cost beyond 8 bytes (call-data length not a multiple of 192: the FIELD quotient is huge)") \
  X(EV_EOPC_NOT_OOG, ZKE_ASSERT, "error_oog_precompile.py:31 gas_left < gas_cost") \
  X(EV_EGUO_CDLEN_UNSAT, ZKE_UNSAT, "error_gas_uint_overflow.py:100 call_context_lookup(CallDataLength) unsat") \
  X(EV_EGUO_CDLEN_AMBIG, ZKE_AMBIG, "error_gas_uint_overflow.py:100 call_context_lookup(CallDataLength) ambiguous") \
  X(EV_EGUO_CDLEN_TYPE, ZKE_ASSERT, "error_gas_uint_overflow.py:100 call_context_lookup(CallDataLength): .value() of a Word") \
  X(EV_EGUO_TXID_UNSAT, ZKE_UNSAT, "error_gas_uint_overflow.py:101 call_context_lookup(TxId) unsat") \
  X(EV_EGUO_TXID_AMBIG, ZKE_AMBIG, "error_gas_uint_overflow.py:101 call_context_lookup(TxId) ambiguous") \
  X(EV_EGUO_TXID_TYPE, ZKE_ASSERT, "error_gas_uint_overflow.py:101 call_context_lookup(TxId): .value() of a Word") \
  X(EV_EGUO_ROOT_UNSAT, ZKE_UNSAT, "error_gas_uint_overflow.py:102 call_context_lookup(IsRoot) unsat") \
  X(EV_EGUO_ROOT_AMBIG, ZKE_AMBIG, "error_gas_uint_overflow.py:102 call_context_lookup(IsRoot) ambiguous") \
  X(EV_EGUO_ROOT_TYPE, ZKE_ASSERT, "error_gas_uint_overflow.py:102 call_context_lookup(IsRoot): .value() of a Word") \
  X(EV_EGUO_BYTE_UNSAT, ZKE_UNSAT, "error_gas_uint_overflow.py:105-108 tx_calldata_lookup(tx_id, idx) unsat") \
  X(EV_EGUO_BYTE_AMBIG, ZKE_AMBIG, "error_gas_uint_overflow.py:105-108 tx_calldata_lookup(tx_id, idx) ambiguous") \
  X(EV_EGUO_BYTE_TYPE, ZKE_ASSERT, "error_gas_uint_overflow.py:105-108 tx_calldata_lookup(tx_id, idx): .value() of a Word") \
  X(EV_EGUO_CMP_RANGE, ZKE_ASSERT, "error_gas_uint_overflow.py:115-137 compare(): an operand beyond 8 bytes (the intrinsic gas itself passed 2^64)") \
  X(EV_EGUO_OPCODE, ZKE_VALUE, "instruction.py:1198-1305 memory_size(opcode) returns None for an opcode without a memory operand -> TypeError (`if is_dynamic_gas:` tests an FQ object, always true)") \
  X(EV_EGUO_POP0_UNSAT, ZKE_UNSAT, "instruction.py:1247-1295 memory_size: stack_pop #0 unsat") \
  X(EV_EGUO_POP0_AMBIG, ZKE_AMBIG, "instruction.py:1247-1295 memory_size: stack_pop #0 ambiguous") \
  X(EV_EGUO_POP1_UNSAT, ZKE_UNSAT, "instruction.py:1247-1295 memory_size: stack_pop #1 unsat") \
  X(EV_EGUO_POP1_AMBIG, ZKE_AMBIG, "instruction.py:1247-1295 memory_size: stack_pop #1 ambiguous") \
  X(EV_EGUO_POP2_UNSAT, ZKE_UNSAT, "instruction.py:1247-1295 memory_size: stack_pop #2 unsat") \
  X(EV_EGUO_POP2_AMBIG, ZKE_AMBIG, "instruction.py:1247-1295 memory_size: stack_pop #2 ambiguous") \
  X(EV_EGUO_POP3_UNSAT, ZKE_UNSAT, "instruction.py:1247-1295 memory_size: stack_pop #3 unsat") \
  X(EV_EGUO_POP3_AMBIG, ZKE_AMBIG, "instruction.py:1247-1295 memory_size: stack_pop #3 ambiguous") \
  X(EV_EGUO_POP4_UNSAT, ZKE_UNSAT, "instruction.py:1247-1295 memory_size: stack_pop #4 unsat") \
  X(EV_EGUO_POP4_AMBIG, ZKE_AMBIG, "instruction.py:1247-1295 memory_size: stack_pop #4 ambiguous") \
  X(EV_EGUO_POP5_UNSAT, ZKE_UNSAT, "instruction.py:1247-1295 memory_size: stack_pop #5 unsat") \
  X(EV_EGUO_POP5_AMBIG, ZKE_AMBIG, "instruction.py:1247-1295 memory_size: stack_pop #5 ambiguous") \
  X(EV_EGUO_POP6_UNSAT, ZKE_UNSAT, "instruction.py:1247-1295 memory_size: stack_pop #6 unsat") \
  X(EV_EGUO_POP6_AMBIG, ZKE_AMBIG, "instruction.py:1247-1295 memory_size: stack_pop #6 ambiguous") \
  X(EV_EGUO_LEN_DOMAIN, ZKE_VALUE, "instruction.py:1310 calc_mem_size64: word_to_fq(length, 31) of a half >= 2^128 -> OverflowError") \
  X(EV_EGUO_LEN_RANGE, ZKE_RANGE, "instruction.py:1310 calc_mem_size64: word_to_fq(length, 31): more than 31 bytes") \
  X(EV_EGUO_OFF_DOMAIN, ZKE_VALUE, "instruction.py:1321 calc_mem_size64_with_uint: word_to_fq(offset, 31) of a half >= 2^128 -> OverflowError") \
  X(EV_EGUO_OFF_RANGE, ZKE_RANGE, "instruction.py:1321 calc_mem_size64_with_uint: word_to_fq(offset, 31): more than 31 bytes") \
  X(EV_EGUO_OFF5_RANGE, ZKE_RANGE, "instruction.py:1325 calc_mem_size64_with_uint: word_to_fq(offset, 5): an offset below 2^64 with more than 5 bytes") \
  X(EV_EGUO_NOT_OVERFLOW, ZKE_ASSERT, "error_gas_uint_overflow.py:160-167 one of the overflow flags is set")

enum zk_evm_constraint { ZK_EVM_CONSTRAINTS(ZK_ENUM_ENTRY) EV_N_CONSTRAINTS };

/* ---------------- copy circuit: src/zkevm_specs/copy_circuit.py:23-130 ----------------------
 * Every gate is `cond * expr == 0` over Fr (util/constraint_system.py:27-46); a row stops at its
 * first failure. */
#define ZK_COPY_CONSTRAINTS(X)                                                             \
  X(CP_BOOL_FIRST, ZKE_ASSERT, "copy_circuit.py:24 is_first boolean")                       \
  X(CP_BOOL_LAST, ZKE_ASSERT, "copy_circuit.py:25 is_last boolean")                         \
  X(CP_FIRST_NEEDS_STEP, ZKE_ASSERT, "copy_circuit.py:27 (1-q_step)*is_first==0")           \
  X(CP_LAST_NOT_STEP, ZKE_ASSERT, "copy_circuit.py:29 q_step*is_last==0")                   \
  X(CP_IS_MEMORY, ZKE_ASSERT, "copy_circuit.py:30 is_memory==(tag==Memory)")                \
  X(CP_IS_BYTECODE, ZKE_ASSERT, "copy_circuit.py:31 is_bytecode==(tag==Bytecode)")          \
  X(CP_IS_TX_CALLDATA, ZKE_ASSERT, "copy_circuit.py:32 is_tx_calldata==(tag==TxCalldata)")  \
  X(CP_IS_TX_LOG, ZKE_ASSERT, "copy_circuit.py:33 is_tx_log==(tag==TxLog)")                 \
  X(CP_IS_RLC_ACC, ZKE_ASSERT, "copy_circuit.py:34 is_rlc_acc==(tag==RlcAcc)")              \
  X(CP_ID_SAME, ZKE_ASSERT, "copy_circuit.py:40 id==rows[2].id unless last two rows")       \
  X(CP_TAG_SAME, ZKE_ASSERT, "copy_circuit.py:41 tag==rows[2].tag")                         \
  X(CP_ADDR_INC, ZKE_ASSERT, "copy_circuit.py:42 addr+1==rows[2].addr")                     \
  X(CP_SRC_END_SAME, ZKE_ASSERT, "copy_circuit.py:43 src_addr_end==rows[2].src_addr_end")   \
  X(CP_RWC, ZKE_ASSERT, "copy_circuit.py:49 rw_counter+rw_diff==next.rw_counter")           \
  X(CP_RWC_INC_LEFT, ZKE_ASSERT, "copy_circuit.py:50 rwc_inc_left-rw_diff==next.rwc_inc_left") \
  X(CP_RLC_ACC_SAME, ZKE_ASSERT, "copy_circuit.py:52 rlc_acc==next.rlc_acc")                \
  X(CP_RWC_INC_LAST, ZKE_ASSERT, "copy_circuit.py:55 last row: rwc_inc_left==rw_diff")      \
  X(CP_RLC_LAST, ZKE_ASSERT, "copy_circuit.py:59 last RlcAcc row: rlc_acc==value")          \
  X(CP_BYTES_LEFT_LAST, ZKE_ASSERT, "copy_circuit.py:65 bytes_left==1 at the last step")    \
  X(CP_BYTES_LEFT_DEC, ZKE_ASSERT, "copy_circuit.py:67 bytes_left==rows[2].bytes_left+1")   \
  X(CP_PAD_VALUE0, ZKE_ASSERT, "copy_circuit.py:69 is_pad*value==0")                        \
  X(CP_LT_RANGE, ZKE_ASSERT, "copy_circuit.py:18-19 lt(): addr / src_addr_end exceed 5 bytes") \
  X(CP_IS_PAD, ZKE_ASSERT, "copy_circuit.py:76-78 is_pad==1-(addr<src_addr_end)")           \
  X(CP_NEXT_NOT_PAD, ZKE_ASSERT, "copy_circuit.py:80 write row is never padding")           \
  X(CP_RW_VALUE_EQ, ZKE_ASSERT, "copy_circuit.py:83 read value==write value unless RlcAcc")  \
  X(CP_FIRST_VALUE_EQ, ZKE_ASSERT, "copy_circuit.py:86 first step: read value==write value") \
  X(CP_RLC_STEP, ZKE_ASSERT, "copy_circuit.py:89 rows[2].value==value*r+rows[1].value")     \
  X(CP_MEM_ID_TYPE, ZKE_ASSERT, "copy_circuit.py:109 id.value(): id is a Word")             \
  X(CP_MEM_UNSAT, ZKE_UNSAT, "copy_circuit.py:108-110 rw_table memory lookup unsat")        \
  X(CP_MEM_AMBIG, ZKE_AMBIG, "copy_circuit.py:108-110 rw_table memory lookup ambiguous")    \
  X(CP_MEM_VALUE_TYPE, ZKE_ASSERT, "copy_circuit.py:110 .value.value(): table value is a Word") \
  X(CP_MEM_VALUE, ZKE_ASSERT, "copy_circuit.py:111 memory byte==row.value")                 \
  X(CP_BC_UNSAT, ZKE_UNSAT, "copy_circuit.py:113-115 bytecode_table lookup unsat")          \
  X(CP_BC_AMBIG, ZKE_AMBIG, "copy_circuit.py:113-115 bytecode_table lookup ambiguous")      \
  X(CP_BC_VALUE, ZKE_ASSERT, "copy_circuit.py:116 bytecode byte==row.value")                \
  X(CP_TX_ID_TYPE, ZKE_ASSERT, "copy_circuit.py:119 id.value(): id is a Word")              \
  X(CP_TX_UNSAT, ZKE_UNSAT, "copy_circuit.py:118-120 tx_table calldata lookup unsat")       \
  X(CP_TX_AMBIG, ZKE_AMBIG, "copy_circuit.py:118-120 tx_table calldata lookup ambiguous")   \
  X(CP_TX_VALUE_TYPE, ZKE_ASSERT, "copy_circuit.py:120 .value.value(): table value is a Word") \
  X(CP_TX_VALUE, ZKE_ASSERT, "copy_circuit.py:121 calldata byte==row.value")                \
  X(CP_LOG_ID_TYPE, ZKE_ASSERT, "copy_circuit.py:127 id.value(): id is a Word")             \
  X(CP_LOG_UNSAT, ZKE_UNSAT, "copy_circuit.py:123-129 rw_table tx-log lookup unsat")        \
  X(CP_LOG_AMBIG, ZKE_AMBIG, "copy_circuit.py:123-129 rw_table tx-log lookup ambiguous")    \
  X(CP_LOG_VALUE_TYPE, ZKE_ASSERT, "copy_circuit.py:129 .value.value(): table value is a Word") \
  X(CP_LOG_VALUE, ZKE_ASSERT, "copy_circuit.py:130 log byte==row.value")

enum zk_copy_constraint { ZK_COPY_CONSTRAINTS(ZK_ENUM_ENTRY) CP_N_CONSTRAINTS };

/* ---------------- state circuit: src/zkevm_specs/state_circuit.py:492-613, 216-488 -----------
 * A row stops at its first failing constraint. */
#define ZK_STATE_CONSTRAINTS(X)                                                            \
  X(ST_TAG_RANGE, ZKE_ASSERT, "state_circuit.py:498 tag in [1,12]")                         \
  X(ST_ID_RANGE, ZKE_ASSERT, "state_circuit.py:499 id in [0,2^28-1]")                       \
  X(ST_FIELD_TAG_RANGE, ZKE_ASSERT, "state_circuit.py:502 field_tag in [0,24]")             \
  X(ST_ADDR_LIMB_RANGE, ZKE_ASSERT, "state_circuit.py:505-506 address limbs are 16-bit")    \
  X(ST_ADDR_LIMBS, ZKE_ASSERT, "state_circuit.py:507-509 address == sum limb_i 2^(16i)")    \
  X(ST_KEY_BYTE_RANGE, ZKE_ASSERT, "state_circuit.py:512-517 (arithmetic.py:20-22) key bytes are 8-bit") \
  X(ST_KEY_BYTES, ZKE_ASSERT, "state_circuit.py:512-517 storage_key == bytes recombined")   \
  X(ST_IS_WRITE_BOOL, ZKE_ASSERT, "state_circuit.py:520 is_write boolean")                  \
  X(ST_PREV_KEY_BYTES, ZKE_VALUE, "state_circuit.py:557-559 int.from_bytes(prev key bytes): a byte >= 256 -> ValueError") \
  X(ST_WITNESS_DOMAIN, ZKE_NOTIMPL, "previous row's keys outside their nominal ranges: packed-key compare outside the supported domain (DESIGN.md)") \
  X(ST_LEX_ORDER, ZKE_ASSERT, "state_circuit.py:552-570 pack(prev) < pack(cur) unless Start") \
  X(ST_READ_CONSISTENCY, ZKE_ASSERT, "state_circuit.py:577-578 read of same keys returns previous value") \
  X(ST_INITIAL_CONSISTENCY, ZKE_ASSERT, "state_circuit.py:580-581 same keys => same initial_value") \
  X(ST_RWC_NONZERO, ZKE_ASSERT, "state_circuit.py:584-585 rw_counter != 0 unless Start")    \
  /* Start :216-236 */                                                                      \
  X(ST_START_FIELD_TAG0, ZKE_ASSERT, "state_circuit.py:218")                                \
  X(ST_START_ADDR0, ZKE_ASSERT, "state_circuit.py:219")                                     \
  X(ST_START_ID0, ZKE_ASSERT, "state_circuit.py:220")                                       \
  X(ST_START_KEY0, ZKE_ASSERT, "state_circuit.py:221")                                      \
  X(ST_START_VALUE_HI0, ZKE_ASSERT, "state_circuit.py:222")                                 \
  X(ST_START_INIT_HI0, ZKE_ASSERT, "state_circuit.py:223")                                  \
  X(ST_START_RWC_INC, ZKE_ASSERT, "state_circuit.py:226 selector*(rwc-prev.rwc-1)==0")      \
  X(ST_START_VALUE0, ZKE_ASSERT, "state_circuit.py:229 value.value()==0")                   \
  X(ST_START_INIT0, ZKE_ASSERT, "state_circuit.py:232 initial_value.value()==0")            \
  X(ST_START_ROOT_SAME, ZKE_ASSERT, "state_circuit.py:235-236")                             \
  /* Memory :240-266 */                                                                     \
  X(ST_MEM_FIELD_TAG0, ZKE_ASSERT, "state_circuit.py:244")                                  \
  X(ST_MEM_KEY0, ZKE_ASSERT, "state_circuit.py:245")                                        \
  X(ST_MEM_VALUE_HI0, ZKE_ASSERT, "state_circuit.py:246")                                   \
  X(ST_MEM_INIT_HI0, ZKE_ASSERT, "state_circuit.py:247")                                    \
  X(ST_MEM_FIRST_READ0, ZKE_ASSERT, "state_circuit.py:253-254 first access read => 0")      \
  X(ST_MEM_ADDR_RANGE, ZKE_ASSERT, "state_circuit.py:257 address <= 2^32-1")                \
  X(ST_MEM_VALUE_BYTE, ZKE_ASSERT, "state_circuit.py:260 value is a byte")                  \
  X(ST_MEM_INIT0, ZKE_ASSERT, "state_circuit.py:263")                                       \
  X(ST_MEM_ROOT_SAME, ZKE_ASSERT, "state_circuit.py:266")                                   \
  /* Stack :270-301 */                                                                      \
  X(ST_STK_FIELD_TAG0, ZKE_ASSERT, "state_circuit.py:275")                                  \
  X(ST_STK_KEY0, ZKE_ASSERT, "state_circuit.py:276")                                        \
  X(ST_STK_FIRST_WRITE, ZKE_ASSERT, "state_circuit.py:285-286 first access is a write")     \
  X(ST_STK_PTR_RANGE, ZKE_ASSERT, "state_circuit.py:290 stack_ptr <= 1023")                 \
  X(ST_STK_PTR_INC, ZKE_ASSERT, "state_circuit.py:293-295 stack_ptr increases by 0 or 1")   \
  X(ST_STK_INIT0, ZKE_ASSERT, "state_circuit.py:298")                                       \
  X(ST_STK_ROOT_SAME, ZKE_ASSERT, "state_circuit.py:301")                                   \
  /* Storage :305-324 */                                                                    \
  X(ST_STO_FIELD_TAG0, ZKE_ASSERT, "state_circuit.py:307")                                  \
  X(ST_STO_MPT_UNSAT, ZKE_UNSAT, "state_circuit.py:313-322 MPT lookup unsat")               \
  X(ST_STO_MPT_AMBIG, ZKE_AMBIG, "state_circuit.py:313-322 MPT lookup ambiguous")           \
  X(ST_STO_ROOT_SAME, ZKE_ASSERT, "state_circuit.py:324")                                   \
  /* CallContext :328-345 */                                                                \
  X(ST_CC_ADDR0, ZKE_ASSERT, "state_circuit.py:330")                                        \
  X(ST_CC_KEY0, ZKE_ASSERT, "state_circuit.py:331")                                         \
  X(ST_CC_FIELD_TAG_RANGE, ZKE_ASSERT, "state_circuit.py:334")                              \
  X(ST_CC_FIRST_READ0, ZKE_ASSERT, "state_circuit.py:338-339")                              \
  X(ST_CC_INIT0, ZKE_ASSERT, "state_circuit.py:342")                                        \
  X(ST_CC_ROOT_SAME, ZKE_ASSERT, "state_circuit.py:345")                                    \
  /* Account :349-380 */                                                                    \
  X(ST_ACC_FIELD_TAG_VALUE, ZKE_VALUE, "state_circuit.py:350 AccountFieldTag(field_tag.n) -> ValueError") \
  X(ST_ACC_ID0, ZKE_ASSERT, "state_circuit.py:353")                                         \
  X(ST_ACC_KEY0, ZKE_ASSERT, "state_circuit.py:354")                                        \
  X(ST_ACC_NONCE_VALUE_HI0, ZKE_ASSERT, "state_circuit.py:356")                             \
  X(ST_ACC_NONCE_INIT_HI0, ZKE_ASSERT, "state_circuit.py:357")                              \
  X(ST_ACC_MPT_UNSAT, ZKE_UNSAT, "state_circuit.py:368-378 MPT lookup unsat")               \
  X(ST_ACC_MPT_AMBIG, ZKE_AMBIG, "state_circuit.py:368-378 MPT lookup ambiguous")           \
  X(ST_ACC_ROOT_SAME, ZKE_ASSERT, "state_circuit.py:380")                                   \
  /* TxRefund :387-402 */                                                                   \
  X(ST_REF_ADDR0, ZKE_ASSERT, "state_circuit.py:389")                                       \
  X(ST_REF_FIELD_TAG0, ZKE_ASSERT, "state_circuit.py:390")                                  \
  X(ST_REF_KEY0, ZKE_ASSERT, "state_circuit.py:391")                                        \
  X(ST_REF_ROOT_SAME, ZKE_ASSERT, "state_circuit.py:394")                                   \
  X(ST_REF_INIT0, ZKE_ASSERT, "state_circuit.py:397")                                       \
  X(ST_REF_FIRST_READ0, ZKE_ASSERT, "state_circuit.py:401-402")                             \
  /* TxAccessListAccount :406-419 */                                                        \
  X(ST_ALA_FIELD_TAG0, ZKE_ASSERT, "state_circuit.py:408")                                  \
  X(ST_ALA_KEY0, ZKE_ASSERT, "state_circuit.py:409")                                        \
  X(ST_ALA_VALUE_HI0, ZKE_ASSERT, "state_circuit.py:410")                                   \
  X(ST_ALA_INIT_HI0, ZKE_ASSERT, "state_circuit.py:411")                                    \
  X(ST_ALA_ROOT_SAME, ZKE_ASSERT, "state_circuit.py:414")                                   \
  X(ST_ALA_FIRST_READ0, ZKE_ASSERT, "state_circuit.py:418-419")                             \
  /* TxAccessListAccountStorage :423-435 */                                                 \
  X(ST_ALS_FIELD_TAG0, ZKE_ASSERT, "state_circuit.py:425")                                  \
  X(ST_ALS_VALUE_HI0, ZKE_ASSERT, "state_circuit.py:426")                                   \
  X(ST_ALS_INIT_HI0, ZKE_ASSERT, "state_circuit.py:427")                                    \
  X(ST_ALS_ROOT_SAME, ZKE_ASSERT, "state_circuit.py:430")                                   \
  X(ST_ALS_FIRST_READ0, ZKE_ASSERT, "state_circuit.py:434-435")                             \
  /* TxLog :439-453 */                                                                      \
  X(ST_LOG_VALUE_HI0, ZKE_ASSERT, "state_circuit.py:446")                                   \
  X(ST_LOG_INIT_HI0, ZKE_ASSERT, "state_circuit.py:447")                                    \
  X(ST_LOG_IS_WRITE, ZKE_ASSERT, "state_circuit.py:450")                                    \
  X(ST_LOG_ROOT_SAME, ZKE_ASSERT, "state_circuit.py:453")                                   \
  /* TxReceipt :460-488 */                                                                  \
  X(ST_RCP_ADDR0, ZKE_ASSERT, "state_circuit.py:465")                                       \
  X(ST_RCP_KEY0, ZKE_ASSERT, "state_circuit.py:466")                                        \
  X(ST_RCP_VALUE_HI0, ZKE_ASSERT, "state_circuit.py:467")                                   \
  X(ST_RCP_INIT_HI0, ZKE_ASSERT, "state_circuit.py:468")                                    \
  X(ST_RCP_STATUS_BOOL, ZKE_ASSERT, "state_circuit.py:471-472")                             \
  X(ST_RCP_TXID_INC, ZKE_ASSERT, "state_circuit.py:476")                                    \
  X(ST_RCP_GAS_INC, ZKE_ASSERT, "state_circuit.py:477-478")                                 \
  X(ST_RCP_FIRST_TXID1, ZKE_ASSERT, "state_circuit.py:481-483")                             \
  X(ST_RCP_TXID_RANGE, ZKE_ASSERT, "state_circuit.py:485")                                  \
  X(ST_RCP_ROOT_SAME, ZKE_ASSERT, "state_circuit.py:488")                                   \
  X(ST_TAG_UNREACHABLE, ZKE_VALUE, "state_circuit.py:612-613 tag 12 has no rules: ValueError")

enum zk_state_constraint { ZK_STATE_CONSTRAINTS(ZK_ENUM_ENTRY) ST_N_CONSTRAINTS };

/* ---------------- exp circuit: src/zkevm_specs/exp_circuit.py:14-97 ------------------------
 * Gates are cond * expr == 0 (util/constraint_system.py); the mul_add_words calls and their
 * range checks run for EVERY row (they are not gated by cs.condition).  A row stops at its
 * first failure. */
#define ZK_EXP_CONSTRAINTS(X)                                                              \
  X(XP_BASE_SAME, ZKE_ASSERT, "exp_circuit.py:18 base == next.base")                        \
  X(XP_A_EQ_NEXT_D, ZKE_ASSERT, "exp_circuit.py:21 a == next.d")                            \
  X(XP_ID_SAME, ZKE_ASSERT, "exp_circuit.py:23 identifier == next.identifier")              \
  X(XP_LAST_BOOL, ZKE_ASSERT, "exp_circuit.py:28 is_step*is_last boolean")                  \
  X(XP_R_BOOL, ZKE_ASSERT, "exp_circuit.py:30 is_step*r boolean")                           \
  X(XP_MUL_TO64, ZKE_VALUE, "arithmetic.py:252-253 to_64s(a|b): half >= 2^128 -> OverflowError") \
  X(XP_MUL_CARRY_LO, ZKE_RANGE, "exp_circuit.py:35 range_check(carry_lo, 9)")               \
  X(XP_MUL_CARRY_HI, ZKE_RANGE, "exp_circuit.py:36 range_check(carry_hi, 9)")               \
  X(XP_EXP_EQ_D, ZKE_ASSERT, "exp_circuit.py:40 exponentiation == d")                       \
  X(XP_C_ZERO, ZKE_ASSERT, "exp_circuit.py:42 c == 0")                                      \
  X(XP_PAR_R_WORD, ZKE_ASSERT, "exp_circuit.py:45 Word.from_lo(r): r >= 2^128")             \
  X(XP_PAR_TO64, ZKE_VALUE, "exp_circuit.py:44-46 to_64s(q): half >= 2^128 -> OverflowError") \
  X(XP_PAR_CARRY_LO, ZKE_RANGE, "exp_circuit.py:47 range_check(carry_lo, 9)")               \
  X(XP_PAR_CARRY_HI, ZKE_RANGE, "exp_circuit.py:48 range_check(carry_hi, 9)")               \
  X(XP_ODD_NEXT_LO, ZKE_ASSERT, "exp_circuit.py:59 odd: next.exponent.lo == exponent.lo - 1") \
  X(XP_ODD_NEXT_HI, ZKE_ASSERT, "exp_circuit.py:61 odd: next.exponent.hi == exponent.hi")   \
  X(XP_ODD_B_BASE, ZKE_ASSERT, "exp_circuit.py:63 odd: b == base")                          \
  X(XP_EVEN_NEXT_LO, ZKE_ASSERT, "exp_circuit.py:72 even: next.exponent.lo == q.lo")        \
  X(XP_EVEN_NEXT_HI, ZKE_ASSERT, "exp_circuit.py:73 even: next.exponent.hi == q.hi")        \
  X(XP_EVEN_A_EQ_B, ZKE_ASSERT, "exp_circuit.py:75 even: a == b")                           \
  X(XP_LAST_EXP_LO2, ZKE_ASSERT, "exp_circuit.py:81 last: exponent.lo == 2")                \
  X(XP_LAST_EXP_HI0, ZKE_ASSERT, "exp_circuit.py:82 last: exponent.hi == 0")                \
  X(XP_LAST_A_BASE, ZKE_ASSERT, "exp_circuit.py:84 last: a == base")                        \
  X(XP_LAST_B_BASE, ZKE_ASSERT, "exp_circuit.py:86 last: b == base")

enum zk_exp_constraint { ZK_EXP_CONSTRAINTS(ZK_ENUM_ENTRY) XP_N_CONSTRAINTS };

/* ---------------- tx circuit, Fr parts: src/zkevm_specs/tx_circuit.py:205-243, 253-289 --------
 * One row per tx_index: SignVerifyChip.verify (keccak-table membership of the RLC of the 64 public
 * key bytes, address == low 20 bytes of the hash, msg_hash == Word(msg_hash_bytes)) and the three
 * copy constraints to the tx-table rows (:278-289).  The ECDSA check itself (tx_circuit.py:147-158)
 * is third-party curve math (eth_keys): its verdict enters as a row flag.  The byte-copy asserts of
 * :209-211 compare two Python copies of the same bytes, stored once here. */
#define ZK_TX_CONSTRAINTS(X)                                                                  \
  X(TX_BYTE_DOMAIN, ZKE_VALUE, "tx_circuit.py:170-172 a `bytes` cell is not < 256 (not representable in the reference)") \
  X(TX_KECCAK_LOOKUP, ZKE_ASSERT, "tx_circuit.py:219-226,57-61 keccak_table.lookup(pub key RLC, 64, hash)") \
  X(TX_ADDRESS, ZKE_ASSERT, "tx_circuit.py:229-232 address == pub_key_hash[-20:]")            \
  X(TX_MSG_HASH, ZKE_ASSERT, "tx_circuit.py:236-239 Word(msg_hash_bytes).select(is_not_padding) == msg_hash") \
  X(TX_ECDSA, ZKE_ASSERT, "tx_circuit.py:242,147-158 ecdsa_verify (third party; verdict supplied as row flag bit 1)") \
  X(TX_ROW_ADDR_TYPE, ZKE_ASSERT, "tx_circuit.py:278 rows[caller].value.value(): the cell is a Word") \
  X(TX_ROW_ADDR, ZKE_ASSERT, "tx_circuit.py:278-281 tx-table CallerAddress == chip address")  \
  X(TX_ROW_HASH_LO, ZKE_ASSERT, "tx_circuit.py:282-285 tx-table TxSignHash.lo == msg_hash.lo") \
  X(TX_ROW_HASH_HI, ZKE_ASSERT, "tx_circuit.py:286-289 tx-table TxSignHash.hi == msg_hash.hi")

enum zk_tx_constraint { ZK_TX_CONSTRAINTS(ZK_ENUM_ENTRY) TX_N_CONSTRAINTS };

/* ---------------- sig circuit, Fr parts: src/zkevm_specs/sig_circuit.py:64-104, 113-123 --------
 * One row per signature: Row.verify.  ECDSA (util/ec.py:109-117, eth_keys) is third party: its
 * boolean verdict enters as row flag bit 1 and is compared with the row's is_valid. */
#define ZK_SIG_CONSTRAINTS(X)                                                                 \
  X(SG_BYTE_DOMAIN, ZKE_VALUE, "sig_circuit.py:36-38 a `bytes` cell is not < 256 (not representable in the reference)") \
  X(SG_SIG_R_COPY, ZKE_ASSERT, "sig_circuit.py:70 sig_r == the ECDSA chip's r")               \
  X(SG_SIG_S_COPY, ZKE_ASSERT, "sig_circuit.py:71 sig_s == the ECDSA chip's s")               \
  X(SG_V_BOOL, ZKE_ASSERT, "sig_circuit.py:74 sig_v in {0, 1}")                               \
  X(SG_KECCAK_LOOKUP, ZKE_ASSERT, "sig_circuit.py:82-88 keccak_table.lookup(pub key RLC, 64, hash)") \
  X(SG_ADDRESS, ZKE_ASSERT, "sig_circuit.py:91-94 recovered_addr == pub_key_hash[-20:]")      \
  X(SG_MSG_HASH, ZKE_ASSERT, "sig_circuit.py:97-100 Word(msg_hash_bytes) == msg_hash")        \
  X(SG_ECDSA_VALID, ZKE_ASSERT, "sig_circuit.py:103-104 ecdsa_chip.verify() == is_valid (third party; verdict = row flag bit 1)")

enum zk_sig_constraint { ZK_SIG_CONSTRAINTS(ZK_ENUM_ENTRY) SG_N_CONSTRAINTS };

/* ---------------- public-inputs circuit: src/zkevm_specs/pi_circuit.py:150-321 ------------------
 * check_row under the loop of verify_circuit (:447-459).  Gates are `selector * polynomial == 0` with
 * inverse witnesses; the three sections after the keccak lookup sit under Python `if selector != 0`. */
#define ZK_PI_CONSTRAINTS(X)                                                                     \
  X(PI_RLC_LAST, ZKE_ASSERT, "pi_circuit.py:162 rpi_bytes_keccakrlc[last] == rpi_bytes[last]")   \
  X(PI_RLC_ACC, ZKE_ASSERT, "pi_circuit.py:165-170 rpi_bytes_keccakrlc[i] == keccak_rand * rpi_bytes_keccakrlc[i+1] + rpi_bytes[i]") \
  X(PI_VALUE_ACC, ZKE_ASSERT, "pi_circuit.py:183-188 rpi_value_lc[i] == rpi_value_lc[i+1] * byte_pow_base + rpi_bytes[i]") \
  X(PI_VALUE_START, ZKE_ASSERT, "pi_circuit.py:191-194 q_rpi_value_start: rpi_value_lc == rpi_bytes") \
  X(PI_KECCAK_WORD, ZKE_ASSERT, "pi_circuit.py:201 rpi_digest_word.select(q): Word((lo, hi)) sanity check, halves < 2^128 (util/arithmetic.py:110-114)") \
  X(PI_KECCAK_LOOKUP, ZKE_ASSERT, "pi_circuit.py:197-203,98-102 keccak_table.lookup(q, q*rlc, q*circuit_len, digest)") \
  X(PI_CD_TXID_INV, ZKE_ASSERT, "pi_circuit.py:208 tx_id * (1 - tx_id_inv * tx_id) == 0")        \
  X(PI_CD_VALUE_INV, ZKE_ASSERT, "pi_circuit.py:209-213 value.lo * (1 - tx_value_lo_inv * value.lo) == 0") \
  X(PI_CD_DIFF_INV, ZKE_ASSERT, "pi_circuit.py:214-216 diff * (1 - tx_id_diff_inv * diff) == 0") \
  X(PI_CD_DEF_TXID, ZKE_ASSERT, "pi_circuit.py:233,240-241 is_tx_id_zero * tx_id")               \
  X(PI_CD_DEF_NEXT_TXID, ZKE_ASSERT, "pi_circuit.py:234 is_tx_id_zero * next.tx_id")             \
  X(PI_CD_DEF_FINAL, ZKE_ASSERT, "pi_circuit.py:235 is_tx_id_zero * is_final")                   \
  X(PI_CD_DEF_GAS, ZKE_ASSERT, "pi_circuit.py:236 is_tx_id_zero * calldata_gas_cost")            \
  X(PI_CD_U16, ZKE_UNSAT, "pi_circuit.py:252-256 lookup(FixedU16Row, tx_id_not_equal_to_next * is_tx_id_next_nonzero * (diff - 1))") \
  X(PI_CD_IDX_SAME, ZKE_ASSERT, "pi_circuit.py:258-260,279 same tx: next.index == index + 1")    \
  X(PI_CD_IDX_NEXT, ZKE_ASSERT, "pi_circuit.py:261-263,280 next tx: next.index == 0")            \
  X(PI_CD_GAS_SAME, ZKE_ASSERT, "pi_circuit.py:264-266,281 same tx: next.gas == gas + gas_cost_next") \
  X(PI_CD_GAS_NEXT, ZKE_ASSERT, "pi_circuit.py:267-271,282 next tx: next.gas == gas_cost_next")  \
  X(PI_CD_GAS_LAST, ZKE_ASSERT, "pi_circuit.py:272,283 padding next: next.gas == 0")             \
  X(PI_CD_FINAL_SAME, ZKE_ASSERT, "pi_circuit.py:273,284 same tx: is_final == 0")                \
  X(PI_CD_FINAL_NEXT, ZKE_ASSERT, "pi_circuit.py:274-276,285 next tx: is_final == 1")            \
  X(PI_CD_START_INDEX, ZKE_ASSERT, "pi_circuit.py:291 calldata start: index == 0")               \
  X(PI_CD_START_GAS, ZKE_ASSERT, "pi_circuit.py:292-294 calldata start: gas == gas_cost")        \
  X(PI_TX_CDL_INV, ZKE_ASSERT, "pi_circuit.py:298 (tag - CallDataLength) * (1 - tx_id_inv * (tag - CallDataLength)) == 0") \
  X(PI_TX_VALUE_INV, ZKE_ASSERT, "pi_circuit.py:299-303 value.lo * (1 - tx_value_lo_inv * value.lo) == 0") \
  X(PI_TX_ZERO_COST, ZKE_ASSERT, "pi_circuit.py:311 CallDataLength == 0 => next row's CallDataGasCost == 0") \
  X(PI_TX_GAS_LOOKUP, ZKE_UNSAT, "pi_circuit.py:312-318 lookup(TxCallDataGasCostAccRow): no row") \
  X(PI_TX_GAS_AMBIG, ZKE_AMBIG, "pi_circuit.py:312-318 lookup(TxCallDataGasCostAccRow): more than one row") \
  X(PI_WD_NEXT_ID, ZKE_ASSERT, "pi_circuit.py:321-322 next.withdrawal.id == withdrawal.id + 1")  \
  X(PI_WD_AMOUNT, ZKE_ASSERT, "pi_circuit.py:323 withdrawal.amount != 0")

enum zk_pi_constraint { ZK_PI_CONSTRAINTS(ZK_ENUM_ENTRY) PI_N_CONSTRAINTS };

/* ---------------- withdrawal circuit: src/zkevm_specs/withdrawal_circuit.py:127-201 -------------------------
 * Per row, in the order verify_circuit evaluates them; the two block-table ids belong to the check after the loop
 * and are reported at row MAX_WITHDRAWALS - 1, behind every id of that row. */
#define ZK_WD_CONSTRAINTS(X)                                                                     \
  X(WD_NEXT_ID, ZKE_ASSERT, "withdrawal_circuit.py:153-158 rows[i+1].withdrawal_id == withdrawal_id + 1 (not on the last row)") \
  X(WD_HASH_WORD, ZKE_ASSERT, "withdrawal_circuit.py:179 withdrawal_hash.select(is_not_padding): Word((lo, hi)) sanity check, halves < 2^128 (util/arithmetic.py:110-114)") \
  X(WD_KECCAK_LOOKUP, ZKE_ASSERT, "withdrawal_circuit.py:169-181,113-117 keccak_table.lookup(q, q*RLC(rlp), q*len(rlp), hash.select(q))") \
  X(WD_MPT_LOOKUP, ZKE_UNSAT, "withdrawal_circuit.py:184-193 mpt_lookup(address, WithdrawalMod / NonExistingAccountProof, Word(id), hash, 0, root, root_prev)") \
  X(WD_BLOCK_LOOKUP, ZKE_UNSAT, "withdrawal_circuit.py:199-201 block_lookup(WithdrawalRoot, rows[MAX-1].root): no row") \
  X(WD_BLOCK_AMBIG, ZKE_AMBIG, "withdrawal_circuit.py:199-201 block_lookup(WithdrawalRoot, rows[MAX-1].root): more than one row")

enum zk_wd_constraint { ZK_WD_CONSTRAINTS(ZK_ENUM_ENTRY) WD_N_CONSTRAINTS };

#endif /* ZK_CONSTRAINTS_H */
