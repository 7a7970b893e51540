/*
 * oracle/withdrawal.c — TEST INFRASTRUCTURE (CPU oracle). Never linked into the product.
 *
 * Restates verify_circuit of the withdrawal circuit, /root/reference/src/zkevm_specs/withdrawal_circuit.py:127-201:
 * for each row below MAX_WITHDRAWALS, in program order, the next-id equality (not on the last row), the Word sanity
 * check of hash.select(is_not_padding), the keccak-table membership of (q, q * RLC(rlp), q * len(rlp), hash), the
 * 12-column MPT lookup; after the loop the block lookup (WithdrawalRoot, rows[MAX-1].root) on field_tag and value.
 * The RLP bytes are built into a buffer (rlp.encode of four integers) and folded by Horner, acc = acc * r + byte.
 * Rows = 8 cells (withdrawal_id, validator_id, address, amount, hash lo, hi, root lo, hi); tables: keccak
 * (is_enabled, input_rlc, input_len, output lo, hi), MPT (address, proof_type, storage_key lo, hi, root lo, hi,
 * root_prev lo, hi, value lo, hi, value_prev lo, hi), block (field_tag, block_number, value lo, hi).  Rows are
 * global rows row_base + local; a row stops at its first failing constraint.  Pinned by tests/golden/withdrawal.npz.
 */
#include "common.h"
#include "lookup.h"

enum { W_ID, W_VALIDATOR, W_ADDRESS, W_AMOUNT, W_HASH_LO, W_HASH_HI, W_ROOT_LO, W_ROOT_HI };
#define WD_TAG_WITHDRAWAL_ROOT 9  /* BlockContextFieldTag.WithdrawalRoot */
#define WD_WITHDRAWAL_MOD 8       /* MPTProofType.WithdrawalMod */
#define WD_NON_EXISTING 4         /* MPTProofType.NonExistingAccountProof */

static const int kWdClass[] = {
#define WD_CLS(id, cls, doc) cls,
    ZK_WD_CONSTRAINTS(WD_CLS)
#undef WD_CLS
};
int orc_wd_n_constraints(void) { return WD_N_CONSTRAINTS; }
int orc_wd_constraint_class(int idx) { return idx >= 0 && idx < WD_N_CONSTRAINTS ? kWdClass[idx] : -1; }

/* rlp.encode of one non-negative integer below 2^256 into out; returns the bytes written */
static int rlp_int(fr_t v, uint8_t* out) {
  uint8_t be[32];
  for (int k = 0; k < 32; k++) be[31 - k] = (uint8_t)(v.l[k / 8] >> (8 * (k % 8)));
  int s = 0;
  while (s < 32 && be[s] == 0) s++;
  const int nb = 32 - s;
  if (nb == 1 && be[31] < 0x80) { out[0] = be[31]; return 1; }
  out[0] = (uint8_t)(0x80 + nb);
  memcpy(out + 1, be + s, (size_t)nb);
  return 1 + nb;
}
/* rlp.encode([id, validator_id, address, amount]) */
static int rlp_row(const fr_t f[4], uint8_t out[140]) {
  uint8_t body[136];
  int n = 0;
  for (int k = 0; k < 4; k++) n += rlp_int(f[k], body + n);
  int h = 0;
  if (n < 56) out[h++] = (uint8_t)(0xC0 + n);
  else { out[h++] = 0xF8; out[h++] = (uint8_t)n; }
  memcpy(out + h, body, (size_t)n);
  return h + n;
}
static fr_t horner(const uint8_t* b, int len, fr_t r) {
  fr_t acc = fr_u64(0);
  for (int i = 0; i < len; i++) acc = fr_add(fr_mul(acc, r), fr_u64(b[i]));
  return acc;
}

int orc_check_withdrawal(const uint64_t* rows, uint64_t n_rows, const uint64_t* keccak, uint64_t n_keccak,
                         const uint64_t* mpt, uint64_t n_mpt, const uint64_t* block, uint64_t n_block, const uint64_t r_l[4],
                         uint64_t max, uint64_t row_begin, uint64_t row_end, uint64_t row_base, uint32_t* first_fail,
                         uint64_t* fail_count) {
  orc_result res_, *res = &res_;
  orc_result_init(res, first_fail, fail_count, WD_N_CONSTRAINTS);
  const uint32_t kk[5] = {0, 1, 2, 3, 4}, mk[12] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11}, bk[3] = {0, 2, 3};
  orc_index kix, mix, bix;
  orc_index_build(&kix, keccak, n_keccak, 5, kk, 5);
  orc_index_build(&mix, mpt, n_mpt, 12, mk, 12);
  orc_index_build(&bix, block, n_block, 4, bk, 3);
  const fr_t r = fr_load(r_l);
#define WK(id, cond) do { if (!(cond)) { orc_fail(res, (id), g); goto next_row; } } while (0)
#define C(c, i) fr_load(ORC_CELL(rows, n_rows, c, i))
  for (uint64_t i = row_begin; i < row_end; i++) {
    const uint64_t g = row_base + i;
    if (g == (max ? max - 1 : 0)) { /* :199-201, after the loop */
      const fr_t key[3] = {fr_u64(WD_TAG_WITHDRAWAL_ROOT), C(W_ROOT_LO, i), C(W_ROOT_HI, i)};
      const int n = orc_lookup(&bix, key, 0);
      REQUIRE(res, WD_BLOCK_LOOKUP, g, n >= 1);
      REQUIRE(res, WD_BLOCK_AMBIG, g, n <= 1);
    }
    if (g >= max) continue;
    {
      const fr_t id = C(W_ID, i), amount = C(W_AMOUNT, i), hlo = C(W_HASH_LO, i), hhi = C(W_HASH_HI, i);
      if (g + 1 < max) WK(WD_NEXT_ID, fr_eq(C(W_ID, i + 1), fr_add(id, fr_u64(1)))); /* :153-158 */
      const fr_t q = fr_u64(fr_is_zero(amount) ? 0 : 1);                           /* :150 */
      const fr_t f[4] = {id, C(W_VALIDATOR, i), C(W_ADDRESS, i), amount};
      uint8_t enc[140];
      const int len = rlp_row(f, enc);
      const fr_t slo = fr_mul(q, hlo), shi = fr_mul(q, hhi);
      WK(WD_HASH_WORD, fr_fits_bits(slo, 128) && fr_fits_bits(shi, 128)); /* :179 Word((lo, hi)) */
      const fr_t kkey[5] = {q, fr_mul(q, horner(enc, len, r)), fr_mul(q, fr_u64((uint64_t)len)), slo, shi};
      WK(WD_KECCAK_LOOKUP, orc_lookup(&kix, kkey, 0) >= 1); /* :169-181 */
      const fr_t proof = fr_add(fr_mul(q, fr_u64(WD_WITHDRAWAL_MOD)), fr_mul(fr_sub(fr_u64(1), q), fr_u64(WD_NON_EXISTING)));
      const fr_t zero = fr_u64(0);
      const fr_t mkey[12] = {C(W_ADDRESS, i), proof, fr_u128(id.l[0], id.l[1]), fr_u128(id.l[2], id.l[3]), C(W_ROOT_LO, i),
                             C(W_ROOT_HI, i), g ? C(W_ROOT_LO, i - 1) : zero, g ? C(W_ROOT_HI, i - 1) : zero, hlo, hhi, zero, zero};
      WK(WD_MPT_LOOKUP, orc_lookup(&mix, mkey, 0) >= 1); /* :184-193 */
    }
  next_row:;
  }
#undef WK
#undef C
  orc_index_free(&kix);
  orc_index_free(&mix);
  orc_index_free(&bix);
  return 0;
}

/* the keccak-table rows withdrawals2witness adds for the given rows (tests: a host-side table for device-assigned
 * witnesses): out = [5][n_rows + 1][4], row 0 the all-zero row, row 1 + i = (1, RLC(rlp(row i)), len, hash lo, hi) */
int orc_wd_keccak_rows(const uint64_t* rows, uint64_t n_rows, const uint64_t r_l[4], uint64_t* out) {
  const fr_t r = fr_load(r_l);
  const uint64_t nk = n_rows + 1;
  memset(out, 0, (size_t)5 * nk * 32);
  for (uint64_t i = 0; i < n_rows; i++) {
    const fr_t f[4] = {fr_load(ORC_CELL(rows, n_rows, W_ID, i)), fr_load(ORC_CELL(rows, n_rows, W_VALIDATOR, i)),
                       fr_load(ORC_CELL(rows, n_rows, W_ADDRESS, i)), fr_load(ORC_CELL(rows, n_rows, W_AMOUNT, i))};
    uint8_t enc[140];
    const int len = rlp_row(f, enc);
    const fr_t v[5] = {fr_u64(1), horner(enc, len, r), fr_u64((uint64_t)len), fr_load(ORC_CELL(rows, n_rows, W_HASH_LO, i)),
                       fr_load(ORC_CELL(rows, n_rows, W_HASH_HI, i))};
    for (int c = 0; c < 5; c++) memcpy(out + ((uint64_t)c * nk + i + 1) * 4, v[c].l, 32);
  }
  return 0;
}
