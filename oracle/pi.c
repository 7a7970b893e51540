/*
 * oracle/pi.c — TEST INFRASTRUCTURE (CPU oracle). Never linked into the product.
 *
 * Restates check_row of the public-inputs circuit, /root/reference/src/zkevm_specs/pi_circuit.py:150-321,
 * under the loop of verify_circuit (:447-459: row_next = rows[(i + 1) % len(rows)]).  Every gate is written
 * as the reference writes it: products over Fr compared with zero, Python `if` on `selector != 0`.
 * Row = 28 cells in the order of pi_circuit.Row (:105-133), Words as (lo, hi), the tx-table and
 * withdrawal-table rows a Row carries flattened behind it:
 *   q_bytes_last, q_tx_table, q_tx_calldata, q_tx_calldata_start, q_rpi_keccak_lookup, q_rpi_value_start,
 *   tx_id_inv, tx_value_lo_inv, tx_id_diff_inv, calldata_gas_cost, is_final, q_withdrawal_table,
 *   rpi_bytes, rpi_bytes_keccakrlc, rpi_value_lc, rpi_digest_word (lo, hi), q_rpi_byte_enable,
 *   tx_table (tx_id, tag, index, value lo, hi), withdrawal_table (id, validator_id, address lo, hi, amount).
 * Tables: keccak (is_enabled, input_rlc, input_len, output lo, hi), set membership of the whole tuple
 * (:78-102); calldata gas cost (tx_id, is_final, gas_cost_acc), lookup() of evm_circuit/table.py:864-884;
 * fixed u16 = the integers 0..65535 (:361).  Parameters: keccak_rand and byte_pow_base (module globals,
 * :834-836) and circuit_len (Witness.circuit_len).  A row stops at its first failing constraint.
 * Pinned by tests/golden/pi_*.npz.
 */
#include "common.h"
#include "lookup.h"

enum { P_Q_BYTES_LAST, P_Q_TX_TABLE, P_Q_TX_CALLDATA, P_Q_TX_CALLDATA_START, P_Q_KECCAK, P_Q_VALUE_START, P_TXID_INV,
       P_VALUE_LO_INV, P_TXID_DIFF_INV, P_CD_GAS, P_IS_FINAL, P_Q_WD, P_BYTES, P_KRLC, P_VALUE_LC, P_DIGEST_LO,
       P_DIGEST_HI, P_Q_BYTE_EN, P_TX_ID, P_TX_TAG, P_TX_INDEX, P_TX_VAL_LO, P_TX_VAL_HI, P_WD_ID, P_WD_VALIDATOR,
       P_WD_ADDR_LO, P_WD_ADDR_HI, P_WD_AMOUNT, PI_COLS };

int orc_check_pi(const uint64_t* rows, uint64_t n_rows, const uint64_t* keccak, uint64_t n_keccak,
                 const uint64_t* gas_tab, uint64_t n_gas, const uint64_t keccak_rand_l[4], const uint64_t byte_base_l[4],
                 const uint64_t circuit_len_l[4], uint64_t row_begin, uint64_t row_end, uint32_t* first_fail,
                 uint64_t* fail_count) {
  orc_result res_, *res = &res_; orc_result_init(res, first_fail, fail_count, PI_N_CONSTRAINTS);
  const uint32_t kk[5] = {0, 1, 2, 3, 4}, gk[3] = {0, 1, 2};
  orc_index kix, gix;
  orc_index_build(&kix, keccak, n_keccak, 5, kk, 5);
  orc_index_build(&gix, gas_tab, n_gas, 3, gk, 3);
  const fr_t keccak_rand = fr_load(keccak_rand_l), byte_base = fr_load(byte_base_l), circuit_len = fr_load(circuit_len_l);
  const fr_t one = fr_u64(1);
#define PK(id, cond) do { if (!(cond)) { orc_fail(res, (id), i); goto next_row; } } while (0)
#define Z(e) fr_is_zero(e)
#define C(c) fr_load(ORC_CELL(rows, n_rows, c, i))
#define N(c) fr_load(ORC_CELL(rows, n_rows, c, j))
#define M fr_mul
  for (uint64_t i = row_begin; i < row_end; i++) {
    const uint64_t j = (i + 1) % n_rows;
    const fr_t en = C(P_Q_BYTE_EN), last = C(P_Q_BYTES_LAST), bytes = C(P_BYTES), krlc = C(P_KRLC), vlc = C(P_VALUE_LC);
    const fr_t vstart = C(P_Q_VALUE_START), qk = C(P_Q_KECCAK);
    /* :162 */
    PK(PI_RLC_LAST, Z(M(M(en, last), fr_sub(krlc, bytes))));
    /* :165-170 */
    PK(PI_RLC_ACC, Z(M(M(en, fr_sub(one, last)), fr_sub(krlc, fr_add(M(N(P_KRLC), keccak_rand), bytes)))));
    /* :183-188 */
    PK(PI_VALUE_ACC, Z(M(M(en, fr_sub(one, vstart)), fr_sub(vlc, fr_add(M(N(P_VALUE_LC), byte_base), bytes)))));
    /* :191-194 */
    PK(PI_VALUE_START, Z(M(M(en, vstart), fr_sub(vlc, bytes))));
    /* :197-203  the selected digest goes through Word((lo, hi)): both halves < 2^128 (util/arithmetic.py:110-114) */
    {
      const fr_t dlo = M(qk, C(P_DIGEST_LO)), dhi = M(qk, C(P_DIGEST_HI));
      PK(PI_KECCAK_WORD, fr_fits_bits(dlo, 128) && fr_fits_bits(dhi, 128));
      fr_t key[5] = {qk, M(qk, krlc), M(qk, circuit_len), dlo, dhi};
      PK(PI_KECCAK_LOOKUP, orc_lookup(&kix, key, 0) >= 1);
    }
    if (!Z(C(P_Q_TX_CALLDATA))) { /* :207-294 */
      const fr_t tx_id = C(P_TX_ID), n_tx_id = N(P_TX_ID), tx_id_inv = C(P_TXID_INV), vlo = C(P_TX_VAL_LO);
      const fr_t vlo_inv = C(P_VALUE_LO_INV), diff_inv = C(P_TXID_DIFF_INV), diff = fr_sub(n_tx_id, tx_id);
      PK(PI_CD_TXID_INV, Z(M(tx_id, fr_sub(one, M(tx_id_inv, tx_id)))));
      PK(PI_CD_VALUE_INV, Z(M(vlo, fr_sub(one, M(vlo_inv, vlo)))));
      PK(PI_CD_DIFF_INV, Z(M(diff, fr_sub(one, M(diff_inv, diff)))));
      const fr_t nz = M(tx_id, tx_id_inv), n_nz = M(n_tx_id, N(P_TXID_INV));
      const fr_t zr = fr_sub(one, nz), n_zr = fr_sub(one, n_nz);
      const fr_t neq = M(diff, diff_inv), eq = fr_sub(one, neq);
      const fr_t b_nz = M(vlo, vlo_inv), nb_nz = M(N(P_TX_VAL_LO), N(P_VALUE_LO_INV));
      const fr_t b_z = fr_sub(one, b_nz), nb_z = fr_sub(one, nb_nz);
      PK(PI_CD_DEF_TXID, Z(M(zr, tx_id)));
      PK(PI_CD_DEF_NEXT_TXID, Z(M(zr, n_tx_id)));
      PK(PI_CD_DEF_FINAL, Z(M(zr, C(P_IS_FINAL))));
      PK(PI_CD_DEF_GAS, Z(M(zr, C(P_CD_GAS))));
      const fr_t gas = fr_add(M(fr_u64(16), b_nz), M(fr_u64(4), b_z));
      const fr_t n_gas = fr_add(M(fr_u64(16), nb_nz), M(fr_u64(4), nb_z));
      /* :250-256 lookup(FixedU16Row): value in 0..65535 */
      PK(PI_CD_U16, fr_fits_bits(M(M(neq, n_nz), fr_sub(diff, one)), 16));
      const fr_t cg = C(P_CD_GAS), ncg = N(P_CD_GAS), fin = C(P_IS_FINAL);
      PK(PI_CD_IDX_SAME, Z(M(nz, M(eq, fr_sub(fr_sub(N(P_TX_INDEX), C(P_TX_INDEX)), one)))));
      PK(PI_CD_IDX_NEXT, Z(M(nz, M(diff, N(P_TX_INDEX)))));
      PK(PI_CD_GAS_SAME, Z(M(nz, M(eq, fr_sub(fr_sub(ncg, cg), n_gas)))));
      PK(PI_CD_GAS_NEXT, Z(M(nz, M(M(n_nz, diff), fr_sub(ncg, n_gas)))));
      PK(PI_CD_GAS_LAST, Z(M(nz, M(n_zr, ncg))));
      PK(PI_CD_FINAL_SAME, Z(M(nz, M(eq, fin))));
      PK(PI_CD_FINAL_NEXT, Z(M(nz, M(diff, fr_sub(fin, one)))));
      const fr_t qs = C(P_Q_TX_CALLDATA_START);
      PK(PI_CD_START_INDEX, Z(M(M(qs, nz), C(P_TX_INDEX))));
      PK(PI_CD_START_GAS, Z(M(M(qs, nz), fr_sub(cg, gas))));
    }
    if (!Z(C(P_Q_TX_TABLE))) { /* :296-318 */
      const fr_t is_cdl = fr_sub(C(P_TX_TAG), fr_u64(8)), inv = C(P_TXID_INV), vlo = C(P_TX_VAL_LO), vinv = C(P_VALUE_LO_INV);
      PK(PI_TX_CDL_INV, Z(M(is_cdl, fr_sub(one, M(inv, is_cdl)))));
      PK(PI_TX_VALUE_INV, Z(M(vlo, fr_sub(one, M(vinv, vlo)))));
      const fr_t cdl_row = fr_sub(one, M(is_cdl, inv)), len_nz = M(vlo, vinv), len_z = fr_sub(one, len_nz);
      const fr_t cost = N(P_TX_VAL_LO);
      PK(PI_TX_ZERO_COST, Z(M(M(cdl_row, len_z), cost)));
      const fr_t qc = M(cdl_row, len_nz);
      fr_t key[3] = {M(C(P_TX_ID), qc), qc, M(cost, qc)};
      const int n = orc_lookup(&gix, key, 0);
      PK(PI_TX_GAS_LOOKUP, n >= 1);
      PK(PI_TX_GAS_AMBIG, n <= 1);
    }
    if (!Z(C(P_Q_WD))) { /* :320-323 */
      if (!Z(N(P_Q_WD))) PK(PI_WD_NEXT_ID, fr_eq(N(P_WD_ID), fr_add(C(P_WD_ID), one)));
      PK(PI_WD_AMOUNT, !Z(C(P_WD_AMOUNT)));
    }
  next_row:;
  }
  orc_index_free(&kix);
  orc_index_free(&gix);
  return 0;
}
